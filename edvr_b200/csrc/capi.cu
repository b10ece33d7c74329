// capi.cu — extern "C" entry points of libedvr_b200.so (see include/edvr_b200.h).
// Host side only validates arguments, fills parameter blocks and launches; no allocation,
// no synchronisation, no global mutable state (the error text is thread-local).
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>

#include "../../include/edvr_b200.h"
#include "common.cuh"
#include "conv_igemm.cuh"
#include "conv_igemm2.cuh"
#include "conv_pair.cuh"
#include "conv_train.cuh"
#include "dcn_backward.cuh"
#include "dcn_f64.cuh"
#include "dcn_fused.cuh"
#include "dcn_site.cuh"
#include "dcn_pair.cuh"
#include "elementwise.cuh"
#include "epilogue.cuh"
#include "selftest.cuh"

using namespace eb;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(EB_ERR_LAUNCH, "%s: %s", what, cudaGetErrorString(e));
    return EB_OK;
}

int num_sms() {
    // per device (a process may drive several GPUs); benign race: every thread computes the same values
    static int n[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    const int slot = dev >= 0 && dev < 64 ? dev : 0;
    if (n[slot] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        n[slot] = v > 0 ? v : 148;
    }
    return n[slot];
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int grid_1d(long long work_items, int block) {
    long long b = (work_items + block - 1) / block;
    long long cap = static_cast<long long>(num_sms()) * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return static_cast<int>(b);
}

int fill_epi(const eb_epilogue_t* e, int H, int W, int cout_packed, EpiParams* o) {
    if (e == nullptr) return fail(EB_ERR_NULLPTR, "epilogue is NULL");
    o->bias = e->bias;
    o->act = e->act;
    o->H = H;
    o->W = W;
    o->res16 = static_cast<const __half*>(e->res16);
    o->res32 = e->res32;
    o->res_pix_stride = e->res_pix_stride;
    o->res_ch_off = e->res_ch_off;
    o->out16 = static_cast<__half*>(e->out16);
    o->out16_pix_stride = e->out16_pix_stride;
    o->out16_ch_off = e->out16_ch_off;
    o->out32 = e->out32;
    o->out32_pix_stride = e->out32_pix_stride;
    o->out32_ch_off = e->out32_ch_off;
    o->out_nchw = e->out_nchw;
    o->nchw_C = e->nchw_C;
    o->out_mode = e->out_mode;
    o->f32_blocked = e->f32_blocked;
    o->bf16 = e->bf16;
    o->res16_wide = (e->res16 && reinterpret_cast<uintptr_t>(e->res16) % 32 == 0 && e->res_pix_stride % 16 == 0 &&
                     e->res_ch_off % 16 == 0) ? 1 : 0;
    if (e->f32_blocked && (e->out_mode != EB_OUT_SAME || (e->out32 && (e->out32_pix_stride % 32 || e->out32_ch_off % 32)) ||
                           (e->res32 && (e->res_pix_stride % 32 || e->res_ch_off % 32)) || e->res16))
        return fail(EB_ERR_UNSUPPORTED, "f32_blocked needs OUT_SAME, C %% 32 == 0, and no fp16 residual");
    if (e->act < EB_ACT_NONE || e->act > EB_ACT_SIGMOID || e->act == 3) return fail(EB_ERR_UNSUPPORTED, "act %d", e->act);
    if (e->out_mode < EB_OUT_SAME || e->out_mode > EB_OUT_STRIDE2)
        return fail(EB_ERR_UNSUPPORTED, "out_mode %d", e->out_mode);
    if (!e->out16 && !e->out32 && !e->out_nchw) return fail(EB_ERR_NULLPTR, "no output pointer");
    if (e->out_mode != EB_OUT_SAME && (!e->out16 || e->out32 || e->out_nchw || e->res16 || e->res32))
        return fail(EB_ERR_UNSUPPORTED, "pixel-shuffle / stride-2 stores support a single fp16 output, no residual");
    if (e->out16 && (!al16(e->out16) || e->out16_pix_stride % 8 || e->out16_ch_off % 8))
        return fail(EB_ERR_ALIGNMENT, "out16 view must be 16-byte aligned");
    if (e->out32 && (!al16(e->out32) || e->out32_pix_stride % 4 || e->out32_ch_off % 4))
        return fail(EB_ERR_ALIGNMENT, "out32 view must be 16-byte aligned");
    if ((e->res16 && (!al16(e->res16) || e->res_pix_stride % 8 || e->res_ch_off % 8)) ||
        (e->res32 && (!al16(e->res32) || e->res_pix_stride % 4 || e->res_ch_off % 4)))
        return fail(EB_ERR_ALIGNMENT, "residual view must be 16-byte aligned");
    if (e->res16 && e->res32) return fail(EB_ERR_UNSUPPORTED, "one residual at most");
    if (e->out_mode == EB_OUT_PIXSHUF2 && cout_packed % 32) return fail(EB_ERR_INVALID_SHAPE, "pixel shuffle needs Cout %% 32 == 0");
    return EB_OK;
}

template <typename KernelT>
int set_smem(KernelT k, int bytes) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return fail(EB_ERR_LAUNCH, "cudaFuncSetAttribute(smem=%d): %s", bytes, cudaGetErrorString(e));
    return EB_OK;
}

}  // namespace

extern "C" {

int eb_version(void) { return 102; }
const char* eb_last_error(void) { return g_err; }

int eb_selftest_umma(const void* A, const void* B, float* D, int N, int K, int variant, void* stream) {
    if (!A || !B || !D) return fail(EB_ERR_NULLPTR, "selftest: null pointer");
    if (N < 32 || N > 256 || N % 32 || K < 16 || K % 16) return fail(EB_ERR_INVALID_SHAPE, "selftest: N=%d K=%d", N, K);
    const int smem = (K / 8) * (128 + N) * 16;
    if (smem > 200 * 1024) return fail(EB_ERR_INVALID_SHAPE, "selftest: K too large");
    if (int rc = set_smem(selftest_umma_kernel, smem)) return rc;
    selftest_umma_kernel<<<1, 128, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(A), static_cast<const __half*>(B), D, N, K, variant);
    return check_launch("selftest_umma");
}

int eb_selftest_mma_rate(int cta_group, int M, int N, int layout, int a_lbo, int a_sbo, int b_lbo, int b_sbo,
                         int kstep_bytes, int reps, unsigned long long* cycles, int* n_ctas, void* stream) {
    if (!cycles || !n_ctas) return fail(EB_ERR_NULLPTR, "mma_rate: null pointer");
    if ((cta_group != 1 && cta_group != 2) || reps < 1) return fail(EB_ERR_INVALID_SHAPE, "mma_rate: cta_group=%d", cta_group);
    MmaRateParams P{M, N, layout, reps, a_lbo, a_sbo, b_lbo, b_sbo, kstep_bytes, cycles};
    const int smem = 96 * 1024;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(num_sms() / cta_group * cta_group);
    cfg.blockDim = dim3(128);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cta_group; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    *n_ctas = static_cast<int>(cfg.gridDim.x);
    cudaError_t e;
    if (cta_group == 2) {
        if (int rc = set_smem(mma_rate_kernel<2>, smem)) return rc;
        e = cudaLaunchKernelEx(&cfg, mma_rate_kernel<2>, P);
    } else {
        if (int rc = set_smem(mma_rate_kernel<1>, smem)) return rc;
        e = cudaLaunchKernelEx(&cfg, mma_rate_kernel<1>, P);
    }
    if (e != cudaSuccess) return fail(EB_ERR_LAUNCH, "mma_rate: %s", cudaGetErrorString(e));
    return check_launch("mma_rate");
}

size_t eb_packed_weight_bytes(int cin, int ktaps, int BN, int n_tiles_n) {
    return static_cast<size_t>(n_tiles_n) * BN * cin * ktaps * 2;
}

int eb_pack_weight(const float* w, int cout, int cin, int ktaps, int BN, int n_tiles_n, void* wpack, void* stream) {
    if (!w || !wpack) return fail(EB_ERR_NULLPTR, "pack_weight: null pointer");
    if (cin % 64 || BN % 32 || BN < 32 || BN > 128 || n_tiles_n < 1 || ktaps < 1 || cout < 1)
        return fail(EB_ERR_INVALID_SHAPE, "pack_weight: cin=%d BN=%d tiles=%d taps=%d", cin, BN, n_tiles_n, ktaps);
    if (cout > BN * n_tiles_n) return fail(EB_ERR_INVALID_SHAPE, "pack_weight: cout exceeds packed rows");
    const long long groups = static_cast<long long>(n_tiles_n) * (cin / 64) * ktaps * 8 * BN;
    pack_weight_kernel<<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        w, cout, cin, ktaps, BN, n_tiles_n, static_cast<__half*>(wpack));
    return check_launch("pack_weight");
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
typedef CUresult (*eb_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                       const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                       CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static eb_encode_tiled_fn tensor_map_encoder() {
    static eb_encode_tiled_fn fn = []() -> eb_encode_tiled_fn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return reinterpret_cast<eb_encode_tiled_fn>(p);
    }();
    return fn;
}

// NHWC fp16 view as a 5-D tensor {8 channels, W, H, pix_stride / 8 K-atoms, images}; box = halo tile of 4 K-atoms
static int encode_halo_map(const ConvSrc& S, int H, int W, int n_images, int taps, CUtensorMap* out) {
    eb_encode_tiled_fn enc = tensor_map_encoder();
    if (!enc) return fail(EB_ERR_UNSUPPORTED, "conv2d_pair: cuTensorMapEncodeTiled unavailable");
    const cuuint64_t ps = static_cast<cuuint64_t>(S.pix_stride);
    const cuuint64_t dims[5] = {8, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), ps / 8, static_cast<cuuint64_t>(n_images)};
    const cuuint64_t strides[4] = {ps * 2, static_cast<cuuint64_t>(W) * ps * 2, 16, static_cast<cuuint64_t>(H) * W * ps * 2};
    const cuuint32_t box[5] = {8, taps == 9 ? CP_RP : CV_TILE, taps == 9 ? CP_RP : CV_TILE, taps == 9 ? 4u : 8u, 1};   // one stage
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<__half*>(S.ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "conv2d_pair: cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r));
    return EB_OK;
}

int eb_pack_weight_pair(const float* w, int cout, int cin, int ktaps, int BN, int n_tiles_n, void* wpack, void* stream) {
    return eb_pack_weight_pair_ex(w, cout, cin, ktaps, BN, n_tiles_n, wpack, 0, stream);
}

int eb_pack_weight_pair_ex(const float* w, int cout, int cin, int ktaps, int BN, int n_tiles_n, void* wpack, int bf16,
                           void* stream) {
    if (!w || !wpack) return fail(EB_ERR_NULLPTR, "pack_weight_pair: null pointer");
    if (cin % 64 || BN % 32 || BN < 32 || BN > 128 || n_tiles_n < 1 || ktaps < 1 || cout < 1)
        return fail(EB_ERR_INVALID_SHAPE, "pack_weight_pair: cin=%d BN=%d tiles=%d taps=%d", cin, BN, n_tiles_n, ktaps);
    if (cout > BN * n_tiles_n) return fail(EB_ERR_INVALID_SHAPE, "pack_weight_pair: cout exceeds packed rows");
    const long long groups = static_cast<long long>(n_tiles_n) * BN * (cin / 8) * ktaps;
    if (bf16)
        pack_weight_pair_kernel<true><<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            w, cout, cin, ktaps, BN, n_tiles_n, static_cast<__half*>(wpack));
    else
        pack_weight_pair_kernel<false><<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            w, cout, cin, ktaps, BN, n_tiles_n, static_cast<__half*>(wpack));
    return check_launch("pack_weight_pair");
}

int eb_pack_weight_pair_dgrad(const float* w, int cout, int cin, int ktaps, int k_channels, int BN, int n_tiles_n, void* wpack,
                              int bf16, void* stream) {
    if (!w || !wpack) return fail(EB_ERR_NULLPTR, "pack_weight_pair_dgrad: null pointer");
    if (k_channels % 64 || k_channels < cout || BN % 32 || BN < 32 || BN > 128 || n_tiles_n < 1 || ktaps < 1 || cin < 1 ||
        BN * n_tiles_n < cin)
        return fail(EB_ERR_INVALID_SHAPE, "pack_weight_pair_dgrad: cout=%d cin=%d K=%d BN=%d tiles=%d", cout, cin, k_channels, BN, n_tiles_n);
    const long long groups = static_cast<long long>(n_tiles_n) * BN * (k_channels / 8) * ktaps;
    if (bf16)
        pack_weight_pair_dgrad_kernel<true><<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            w, cout, cin, ktaps, k_channels, BN, n_tiles_n, static_cast<__half*>(wpack));
    else
        pack_weight_pair_dgrad_kernel<false><<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            w, cout, cin, ktaps, k_channels, BN, n_tiles_n, static_cast<__half*>(wpack));
    return check_launch("pack_weight_pair_dgrad");
}

int eb_conv2d_pair_supported(int cin, int ksize, int BN, int n_tiles_n) {
    if (cin < 64 || cin % 64 || (ksize != 3 && ksize != 1) || BN % 32 || BN < 32 || BN > 128 || n_tiles_n < 1) return 0;
    if (n_tiles_n > num_sms() / 2 || tensor_map_encoder() == nullptr) return 0;
    // 1: each CTA keeps its half of the weights resident in shared memory; 2: weights stream with the activation stages
    // (always for 1x1 layers: 64-channel stages, no halo)
    if (ksize == 1) return getenv("EDVR_B200_PAIR_1X1_OFF") ? 0 : 2;
    return static_cast<long long>(cin) * ksize * ksize * (BN / 2) * 2 <= CP_W_BYTES ? 1 : 2;
}

static bool conv_force_v1() {
    const char* e = getenv("EDVR_B200_CONV_V1");     // A/B switch for profiling; read-only, no mutable state
    return e != nullptr && e[0] == '1';
}

static bool conv_force_v2() {
    const char* e = getenv("EDVR_B200_CONV_V2");
    return e != nullptr && e[0] == '1';
}

static int launch_conv(const ConvParams& P, cudaStream_t st) {
    if (P.N == 0) return EB_OK;
    if (P.epi.bf16) return fail(EB_ERR_UNSUPPORTED, "conv2d: bf16 operands are served by the CTA-pair kernel only (eb_conv2d_pair)");
    // epilogue kind of the transposed kernel (conv_igemm2.cuh); combinations it does not cover use the generic kernel
    int ek = -1;
    // measured on B200 (profiles/r01_conv_stats_*): the channel-major kernel wins when the K loop is long
    // (Cin >= 256: the per-tile epilogue is amortised) and for the PixelShuffle store; the pixel-major kernel
    // (16-byte stores, 8x fewer store instructions per thread) wins elsewhere.
    const int cin_total = P.src[0].C + (P.nsrc > 1 ? P.src[1].C : 0);
    const bool prefer_v2 = conv_force_v2() || (P.taps == 9 && (cin_total >= 256 || P.epi.out_mode == OUT_PIXSHUF2)) || P.stats != nullptr;
    if (P.BN == 128 && P.epi.out_nchw == nullptr && !P.epi.f32_blocked && !conv_force_v1() && prefer_v2) {
        const EpiParams& e = P.epi;
        if (e.out_mode == OUT_PIXSHUF2) ek = EK_PIXSHUF;
        else if (e.out_mode == OUT_STRIDE2) ek = EK_STRIDE2;
        else if (e.out32 || e.res32) { if (!e.res16) ek = EK_F32; }
        else if (e.out16) ek = EK_PLAIN;
    }
    if (ek >= 0) {
        const long long tiles2 = static_cast<long long>(P.N) * ((P.H + C2_TH - 1) / C2_TH) * ((P.W + C2_TW - 1) / C2_TW) * P.n_tiles_n;
        const int grid2 = static_cast<int>(tiles2 < num_sms() ? tiles2 : num_sms());
        const bool halo = P.taps == 9, stats = P.stats != nullptr;
#define EB_LAUNCH_C2(HALO_, EK_, ST_, PS_)                                                             \
        do {                                                                                           \
            if (int rc = set_smem(conv_igemm2_kernel<HALO_, EK_, ST_, PS_>, C2_SMEM_BYTES)) return rc; \
            conv_igemm2_kernel<HALO_, EK_, ST_, PS_><<<grid2, C2_THREADS, C2_SMEM_BYTES, st>>>(P);     \
        } while (0)
#define EB_DISPATCH_C2(EK_)                                                                            \
        do {                                                                                           \
            if (stats && halo) EB_LAUNCH_C2(1, EK_, true, 0);                                          \
            else if (halo && ps == 128) EB_LAUNCH_C2(1, EK_, false, 128);                              \
            else if (halo && ps == 256) EB_LAUNCH_C2(1, EK_, false, 256);                              \
            else if (halo) EB_LAUNCH_C2(1, EK_, false, 0);                                             \
            else if (ps == 128) EB_LAUNCH_C2(0, EK_, false, 128);                                      \
            else EB_LAUNCH_C2(0, EK_, false, 0);                                                       \
        } while (0)
        // compile-time pixel stride when every tensor the epilogue touches agrees on it
        int ps = P.epi.out16 ? P.epi.out16_pix_stride : (P.epi.out32 ? P.epi.out32_pix_stride : 0);
        if ((P.epi.out32 && P.epi.out32_pix_stride != ps) || ((P.epi.res16 || P.epi.res32) && P.epi.res_pix_stride != ps)) ps = 0;
        switch (ek) {
            case EK_PLAIN: EB_DISPATCH_C2(EK_PLAIN); break;
            case EK_F32: EB_DISPATCH_C2(EK_F32); break;
            case EK_PIXSHUF: EB_DISPATCH_C2(EK_PIXSHUF); break;
            default: EB_DISPATCH_C2(EK_STRIDE2); break;
        }
#undef EB_DISPATCH_C2
#undef EB_LAUNCH_C2
        return check_launch("conv_igemm2");
    }
    const long long tiles = static_cast<long long>(P.N) * ((P.H + 15) / 16) * ((P.W + 15) / 16) * P.n_tiles_n;
    const int grid = static_cast<int>(tiles < num_sms() ? tiles : num_sms());
    // pixel-major kernel: compact instantiations for the common epilogues, generic one for everything else
    int ek1 = EK_GENERIC;
    {
        const EpiParams& e = P.epi;
        const bool plain_out = e.out16 && !e.out32 && !e.res32 && !e.out_nchw;
        if (e.out_mode == OUT_PIXSHUF2) ek1 = EK_PIXSHUF;
        else if (e.out_mode == OUT_STRIDE2) ek1 = EK_STRIDE2;
        else if (plain_out) ek1 = EK_PLAIN;
        else if ((e.out32 || e.res32) && !e.res16 && !e.out_nchw) ek1 = EK_F32;
    }
#define EB_LAUNCH_C1(HALO_, EK_)                                                                       \
    do {                                                                                               \
        if (int rc = set_smem(conv_igemm_kernel<HALO_, EK_>, CV_SMEM_BYTES)) return rc;                \
        conv_igemm_kernel<HALO_, EK_><<<grid, CV_THREADS, CV_SMEM_BYTES, st>>>(P);                     \
    } while (0)
#define EB_DISPATCH_C1(HALO_)                                                                          \
    do {                                                                                               \
        switch (ek1) {                                                                                 \
            case EK_PLAIN: EB_LAUNCH_C1(HALO_, EK_PLAIN); break;                                       \
            case EK_F32: EB_LAUNCH_C1(HALO_, EK_F32); break;                                           \
            case EK_PIXSHUF: EB_LAUNCH_C1(HALO_, EK_PIXSHUF); break;                                   \
            case EK_STRIDE2: EB_LAUNCH_C1(HALO_, EK_STRIDE2); break;                                   \
            default: EB_LAUNCH_C1(HALO_, EK_GENERIC); break;                                           \
        }                                                                                              \
    } while (0)
    if (P.taps == 9) EB_DISPATCH_C1(1); else EB_DISPATCH_C1(0);
#undef EB_DISPATCH_C1
#undef EB_LAUNCH_C1
    return check_launch("conv_igemm");
}

static int build_conv_params(const char* who, const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize,
                             const void* wpack, int BN, int n_tiles_n, const eb_epilogue_t* epi, bool bias_in_smem_table,
                             ConvParams* out) {
    if (!srcs || !wpack) return fail(EB_ERR_NULLPTR, "%s: null pointer", who);
    if (nsrc < 1 || nsrc > 2) return fail(EB_ERR_UNSUPPORTED, "%s: nsrc=%d", who, nsrc);
    if (ksize != 1 && ksize != 3) return fail(EB_ERR_UNSUPPORTED, "%s: ksize=%d", who, ksize);
    if (N < 0 || H < 1 || W < 1) return fail(EB_ERR_INVALID_SHAPE, "%s: N=%d H=%d W=%d", who, N, H, W);
    if (BN % 32 || BN < 32 || BN > 128 || n_tiles_n < 1 ||
        (bias_in_smem_table && epi && epi->bias && BN * n_tiles_n > CV_MAX_COUT))
        return fail(EB_ERR_INVALID_SHAPE, "%s: BN=%d n_tiles_n=%d", who, BN, n_tiles_n);
    if (!al16(wpack)) return fail(EB_ERR_ALIGNMENT, "%s: wpack must be 16-byte aligned", who);
    ConvParams& P = *out;
    memset(&P, 0, sizeof(P));
    for (int i = 0; i < nsrc; ++i) {
        const eb_src_t& s = srcs[i];
        if (!s.ptr) return fail(EB_ERR_NULLPTR, "%s: src %d null", who, i);
        if (s.C < 64 || s.C % 64) return fail(EB_ERR_INVALID_SHAPE, "%s: src %d C=%d (multiple of 64)", who, i, s.C);
        if (!al16(s.ptr) || s.pix_stride % 8 || s.ch_off % 8 || s.pix_stride < s.C + s.ch_off)
            return fail(EB_ERR_ALIGNMENT, "%s: src %d view (stride %d, off %d)", who, i, s.pix_stride, s.ch_off);
        if (s.div < 1) return fail(EB_ERR_INVALID_SHAPE, "%s: src %d div=%d", who, i, s.div);
        P.src[i].ptr = static_cast<const __half*>(s.ptr);
        P.src[i].C = s.C; P.src[i].pix_stride = s.pix_stride; P.src[i].ch_off = s.ch_off;
        P.src[i].div = s.div; P.src[i].mul = s.mul; P.src[i].keep = s.keep; P.src[i].add = s.add;
    }
    P.nsrc = nsrc; P.N = N; P.H = H; P.W = W; P.taps = ksize * ksize; P.BN = BN; P.n_tiles_n = n_tiles_n;
    P.wpack = static_cast<const __half*>(wpack);
    if (int rc = fill_epi(epi, H, W, BN * n_tiles_n, &P.epi)) return rc;
    { const char* e = getenv("EDVR_B200_DBG"); P.dbg = e != nullptr ? atoi(e) : 0; }   // profiling switches (wrong results)
    return EB_OK;
}

int eb_conv2d(const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize, const void* wpack, int BN,
              int n_tiles_n, const eb_epilogue_t* epi, void* stream) {
    return eb_conv2d_stats(srcs, nsrc, N, H, W, ksize, wpack, BN, n_tiles_n, epi, nullptr, stream);
}

int eb_conv2d_stats(const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize, const void* wpack, int BN,
                    int n_tiles_n, const eb_epilogue_t* epi, unsigned long long* stats, void* stream) {
    ConvParams P;
    if (int rc = build_conv_params("conv2d", srcs, nsrc, N, H, W, ksize, wpack, BN, n_tiles_n, epi, true, &P)) return rc;
    P.stats = stats;
    return launch_conv(P, static_cast<cudaStream_t>(stream));
}

// CTA-pair kernel with shared-memory-resident weights (conv_pair.cuh); `wpair` comes from eb_pack_weight_pair.
int eb_conv2d_pair(const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize, const void* wpair, int BN,
                   int n_tiles_n, const eb_epilogue_t* epi, void* stream) {
    ConvParams P;
    if (int rc = build_conv_params("conv2d_pair", srcs, nsrc, N, H, W, ksize, wpair, BN, n_tiles_n, epi, false, &P)) return rc;
    const int cin = P.src[0].C + (nsrc > 1 ? P.src[1].C : 0);
    const int mode = eb_conv2d_pair_supported(cin, ksize, BN, n_tiles_n);
    if (!mode) return fail(EB_ERR_UNSUPPORTED, "conv2d_pair: cin=%d k=%d BN=%d tiles=%d", cin, ksize, BN, n_tiles_n);
    const bool resident = mode == 1 && !(P.dbg & 128);
    if (N == 0) return EB_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long pair_tiles = static_cast<long long>(N) * ((H + 15) / 16) * (((W + 15) / 16 + 1) / 2);
    long long want = pair_tiles * n_tiles_n;
    const int max_clusters = num_sms() / 2;
    int nclusters = static_cast<int>(want < max_clusters ? want : max_clusters);
    nclusters = nclusters / n_tiles_n * n_tiles_n;
    if (nclusters < n_tiles_n) nclusters = n_tiles_n;
    int ek1 = EK_GENERIC;
    {
        const EpiParams& e = P.epi;
        const bool plain_out = e.out16 && !e.out32 && !e.res32 && !e.out_nchw;
        if (e.out_mode == OUT_PIXSHUF2) ek1 = EK_PIXSHUF;
        else if (e.out_mode == OUT_STRIDE2) ek1 = EK_STRIDE2;
        else if (plain_out) ek1 = EK_PLAIN;
        else if ((e.out32 || e.res32) && !e.res16 && !e.out_nchw) ek1 = EK_F32;
    }
    PairParams PP;
    PP.c = P;
    for (int i = 0; i < nsrc; ++i) {
        const ConvSrc& S = P.src[i];
        const int last = N - 1;       // largest source image index the kernel can ask for
        const int n_images = (last / S.div) * S.mul + ((last < S.div ? last : S.div - 1)) * (S.keep > 0 ? S.keep : 0) + S.add + 1;
        if (int rc = encode_halo_map(S, H, W, n_images < 1 ? 1 : n_images, P.taps, &PP.tmap[i])) return rc;
    }
    if (nsrc == 1) PP.tmap[1] = PP.tmap[0];
    PP.tmap_w = PP.tmap[0];
    if (!resident) {
        // packed weights as rows of 256 fp16; one box = the (BN/2) x 9 x 32 slice one CTA needs for one 32-channel chunk
        eb_encode_tiled_fn enc = tensor_map_encoder();
        const cuuint64_t total = static_cast<cuuint64_t>(n_tiles_n) * BN * cin * P.taps;     // fp16 elements
        const cuuint64_t dims[2] = {256, total / 256};
        const cuuint64_t strides[1] = {512};
        const cuuint32_t box[2] = {256, static_cast<cuuint32_t>((P.taps == 9 ? 9 * 4 : 8) * (BN / 2) * 16 / 512)};   // one stage
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = enc(&PP.tmap_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(P.wpack), dims, strides, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "conv2d_pair: weight tensor map failed (%d)", static_cast<int>(r));
    }
    // fp16 NHWC output through TMA when the epilogue writes it pixel-for-pixel (plain / fp32-stream kinds)
    PP.tma_out = 0;
    PP.tmap_out = PP.tmap[0];
    if ((ek1 == EK_PLAIN || ek1 == EK_F32) && P.epi.out16 != nullptr && !(P.dbg & 64)) {
        eb_encode_tiled_fn enc = tensor_map_encoder();
        const cuuint64_t ps = static_cast<cuuint64_t>(P.epi.out16_pix_stride);
        const cuuint64_t dims[4] = {ps, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[3] = {ps * 2, static_cast<cuuint64_t>(W) * ps * 2, static_cast<cuuint64_t>(H) * W * ps * 2};
        const cuuint32_t box[4] = {32, 8, 4, 1};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult r = enc(&PP.tmap_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, P.epi.out16, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "conv2d_pair: output tensor map failed (%d)", static_cast<int>(r));
        PP.tma_out = 1;
    } else if (ek1 == EK_PIXSHUF && P.epi.out16 != nullptr && !(P.dbg & 64)) {
        // PixelShuffle(2) store: the output is [N, 2H, 2W, Cout/4]; one box = 8 channels of the 16 x 8 output pixels of a warp
        eb_encode_tiled_fn enc = tensor_map_encoder();
        const cuuint64_t ps = static_cast<cuuint64_t>(P.epi.out16_pix_stride);
        const cuuint64_t W2 = 2ull * W, H2 = 2ull * H;
        const cuuint64_t dims[4] = {ps, W2, H2, static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[3] = {ps * 2, W2 * ps * 2, H2 * W2 * ps * 2};
        const cuuint32_t box[4] = {8, 16, 8, 1};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult r = enc(&PP.tmap_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, P.epi.out16, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "conv2d_pair: pixel-shuffle tensor map failed (%d)", static_cast<int>(r));
        PP.tma_out = 1;
    }
    if (P.epi.bf16 && !(ek1 == EK_PLAIN && PP.tma_out && !P.epi.res16))
        return fail(EB_ERR_UNSUPPORTED, "conv2d_pair: bf16 needs the plain NHWC output (no residual, no index map)");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * nclusters);
    cfg.blockDim = dim3(CP_THREADS);
    cfg.dynamicSmemBytes = P.taps == 1 ? CP_SMEM_BYTES_1X1 : resident ? CP_SMEM_BYTES : CP_SMEM_BYTES_STREAM;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;      // see pdl_wait() in conv_pair.cuh
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = getenv("EDVR_B200_NO_PDL") ? 1 : 2;
    cudaError_t err = cudaSuccess;
#define EB_LAUNCH_CP(EK_, TO_)                                                                         \
    do {                                                                                               \
        if (P.taps == 1) {                                                                             \
            if (int rc = set_smem(conv_pair_kernel<EK_, TO_, false, 1>, CP_SMEM_BYTES_1X1)) return rc; \
            err = cudaLaunchKernelEx(&cfg, conv_pair_kernel<EK_, TO_, false, 1>, PP);                  \
        } else if (resident) {                                                                         \
            if (int rc = set_smem(conv_pair_kernel<EK_, TO_, true>, CP_SMEM_BYTES)) return rc;         \
            err = cudaLaunchKernelEx(&cfg, conv_pair_kernel<EK_, TO_, true>, PP);                      \
        } else {                                                                                       \
            if (int rc = set_smem(conv_pair_kernel<EK_, TO_, false>, CP_SMEM_BYTES_STREAM)) return rc; \
            err = cudaLaunchKernelEx(&cfg, conv_pair_kernel<EK_, TO_, false>, PP);                     \
        }                                                                                              \
    } while (0)
    switch (ek1) {
        case EK_PLAIN: if (PP.tma_out) EB_LAUNCH_CP(EK_PLAIN, true); else EB_LAUNCH_CP(EK_PLAIN, false); break;
        case EK_F32: if (PP.tma_out) EB_LAUNCH_CP(EK_F32, true); else EB_LAUNCH_CP(EK_F32, false); break;
        case EK_PIXSHUF: if (PP.tma_out) EB_LAUNCH_CP(EK_PIXSHUF, true); else EB_LAUNCH_CP(EK_PIXSHUF, false); break;
        case EK_STRIDE2: EB_LAUNCH_CP(EK_STRIDE2, false); break;
        default: EB_LAUNCH_CP(EK_GENERIC, false); break;
    }
#undef EB_LAUNCH_CP
    if (err != cudaSuccess) return fail(EB_ERR_LAUNCH, "conv2d_pair: %s", cudaGetErrorString(err));
    return check_launch("conv_pair");
}

// ---- training step: weight gradient of a dense 3x3 (pad 1) / 1x1 convolution (conv_train.cuh)
namespace {
struct WgradGeo { int Hp, Wp, margin, BN, splits, steps_per_split; long long body, Ppad, k_steps; size_t rowsA, a_bytes, b_bytes, p_bytes; int copies; };
WgradGeo wgrad_geo(int N, int H, int W, int Cin, int Cout, int ksize) {
    WgradGeo g;
    g.Hp = H + 2; g.Wp = (W + 2 + 7) / 8 * 8;
    g.margin = (g.Wp + 8 + 63) / 64 * 64;
    g.body = (static_cast<long long>(N) * g.Hp * g.Wp + 63) / 64 * 64;
    g.Ppad = g.body + 2 * g.margin;
    g.rowsA = static_cast<size_t>((Cout + 127) / 128) * 128;
    g.copies = ksize == 3 ? 3 : 1;
    g.a_bytes = (g.rowsA * g.Ppad * 2 + 255) / 256 * 256;
    g.b_bytes = (static_cast<size_t>(g.copies) * Cin * g.Ppad * 2 + 255) / 256 * 256;
    g.BN = Cin % 128 == 0 ? 128 : (Cin % 64 == 0 ? 64 : (Cin % 32 == 0 ? 32 : 0));
    g.k_steps = g.body / 64;
    const int tiles = g.BN ? ksize * ksize * (Cin / g.BN) * static_cast<int>(g.rowsA / 128) : 1;
    long long splits = (2LL * 148) / tiles;                      // one wave of 2 CTAs per SM; at least 24 K steps per split
    if (splits > g.k_steps / 24) splits = g.k_steps / 24;        // (prologue + 64 KB partial tile amortised over >= 1.5K pixels)
    if (splits < 1) splits = 1;
    g.steps_per_split = static_cast<int>((g.k_steps + splits - 1) / splits);
    g.splits = static_cast<int>((g.k_steps + g.steps_per_split - 1) / g.steps_per_split);
    g.p_bytes = (static_cast<size_t>(g.splits) * ksize * ksize * Cin * g.rowsA * 4 + 255) / 256 * 256;
    return g;
}
}  // namespace

size_t eb_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int ksize) {
    const WgradGeo g = wgrad_geo(N, H, W, Cin, Cout, ksize);
    return g.a_bytes + g.b_bytes + g.p_bytes;
}

int eb_conv_wgrad(const void* x, int x_pix_stride, int x_ch_off, const void* gy, int gy_pix_stride, int gy_ch_off, int N,
                  int H, int W, int Cin, int Cout, int ksize, int bf16, float scale, float* grad_weight, float* grad_bias,
                  void* workspace, size_t workspace_bytes, void* stream) {
    if (!x || !gy || !grad_weight) return fail(EB_ERR_NULLPTR, "conv_wgrad: null pointer");
    if (N < 1 || H < 1 || W < 1 || Cout < 1 || Cin < 32 || (ksize != 1 && ksize != 3))
        return fail(EB_ERR_INVALID_SHAPE, "conv_wgrad: N=%d H=%d W=%d Cin=%d Cout=%d k=%d", N, H, W, Cin, Cout, ksize);
    const WgradGeo g = wgrad_geo(N, H, W, Cin, Cout, ksize);
    const int BN = g.BN;
    if (!BN) return fail(EB_ERR_UNSUPPORTED, "conv_wgrad: Cin=%d must be a multiple of 32", Cin);
    if (x_pix_stride < x_ch_off + Cin || gy_pix_stride < gy_ch_off + Cout) return fail(EB_ERR_INVALID_SHAPE, "conv_wgrad: views");
    const size_t need = g.a_bytes + g.b_bytes + g.p_bytes;
    if (!workspace || workspace_bytes < need) return fail(EB_ERR_WORKSPACE, "conv_wgrad: workspace %zu < %zu", workspace_bytes, need);
    if (!al16(workspace)) return fail(EB_ERR_ALIGNMENT, "conv_wgrad: workspace must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint16_t* gyT = static_cast<uint16_t*>(workspace);
    uint16_t* xT = reinterpret_cast<uint16_t*>(static_cast<uint8_t*>(workspace) + g.a_bytes);
    float* partial = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + g.a_bytes + g.b_bytes);
    if (cudaMemsetAsync(workspace, 0, g.a_bytes + g.b_bytes, st) != cudaSuccess) return fail(EB_ERR_LAUNCH, "conv_wgrad: memset");
    const long long copy_stride = static_cast<long long>(Cin) * g.Ppad;
    {
        dim3 block(32, 8);
        const int rows_g = grad_bias ? CT_ROWS : 1;
        dim3 grid_g((W + 31) / 32, static_cast<unsigned>((H + rows_g - 1) / rows_g), N * ((Cout + 31) / 32));
        dim3 grid_x((W + 31) / 32, static_cast<unsigned>(H), N * ((Cin + 31) / 32));
        if (bf16) {
            nhwc_to_cmajor_pad_kernel<true><<<grid_g, block, 0, st>>>(static_cast<const uint16_t*>(gy), gy_pix_stride, gy_ch_off, Cout,
                                                                      H, W, gyT, 0, g.Ppad, g.Hp, g.Wp, g.margin, 1, grad_bias, rows_g);
            nhwc_to_cmajor_pad_kernel<true><<<grid_x, block, 0, st>>>(static_cast<const uint16_t*>(x), x_pix_stride, x_ch_off, Cin, H,
                                                                      W, xT, copy_stride, g.Ppad, g.Hp, g.Wp, g.margin, g.copies, nullptr, 1);
        } else {
            nhwc_to_cmajor_pad_kernel<false><<<grid_g, block, 0, st>>>(static_cast<const uint16_t*>(gy), gy_pix_stride, gy_ch_off, Cout,
                                                                       H, W, gyT, 0, g.Ppad, g.Hp, g.Wp, g.margin, 1, grad_bias, rows_g);
            nhwc_to_cmajor_pad_kernel<false><<<grid_x, block, 0, st>>>(static_cast<const uint16_t*>(x), x_pix_stride, x_ch_off, Cin, H,
                                                                       W, xT, copy_stride, g.Ppad, g.Hp, g.Wp, g.margin, g.copies, nullptr, 1);
        }
        if (int rc = check_launch("conv_wgrad transposes")) return rc;
    }
    const int taps = ksize * ksize;
    if (int rc = set_smem(conv_wgrad_kernel, CW_SMEM_BYTES)) return rc;
    const unsigned m_tiles = static_cast<unsigned>(g.rowsA / 128);
    dim3 grid(taps * (Cin / BN), m_tiles, static_cast<unsigned>(g.splits));
    eb_encode_tiled_fn enc = tensor_map_encoder();
    if (!enc) return fail(EB_ERR_UNSUPPORTED, "conv_wgrad: cuTensorMapEncodeTiled unavailable");
    WgradParams WP;
    memset(&WP, 0, sizeof(WP));
    {
        // channel-major rows [rows][Ppad] as {8 elements, rows, Ppad / 8 atoms}: a box {8, R, 8} is one 64-pixel K step in the
        // no-swizzle K-major operand layout ([K atom][row][16 B])
        const cuuint64_t atoms = static_cast<cuuint64_t>(g.Ppad / 8);
        const cuuint32_t estr[3] = {1, 1, 1};
        const cuuint64_t strides[2] = {static_cast<cuuint64_t>(g.Ppad) * 2, 16};
        const cuuint64_t dims_a[3] = {8, static_cast<cuuint64_t>(g.rowsA), atoms};
        const cuuint32_t box_a[3] = {8, 128, 8};
        CUresult r = enc(&WP.tmap_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, gyT, dims_a, strides, box_a, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "conv_wgrad: tensor map A failed (%d)", static_cast<int>(r));
        const cuuint64_t dims_b[3] = {8, static_cast<cuuint64_t>(g.copies) * Cin, atoms};
        const cuuint32_t box_b[3] = {8, static_cast<cuuint32_t>(BN), 8};
        r = enc(&WP.tmap_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, xT, dims_b, strides, box_b, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "conv_wgrad: tensor map B failed (%d)", static_cast<int>(r));
    }
    WP.partial = partial; WP.Cin = Cin; WP.taps = taps; WP.BN = BN; WP.Wp = g.Wp; WP.steps_per_split = g.steps_per_split;
    WP.ab_fmt = bf16 ? 1 : 0; WP.k_begin = g.margin; WP.k_steps = g.k_steps;
    conv_wgrad_kernel<<<grid, CW_THREADS, CW_SMEM_BYTES, st>>>(WP);
    if (int rc = check_launch("conv_wgrad")) return rc;
    const long long total = static_cast<long long>(taps) * Cout * Cin;
    conv_wgrad_reduce_kernel<<<grid_1d(total, 256), 256, 0, st>>>(partial, grad_weight, Cout, Cin, taps, BN, static_cast<int>(m_tiles),
                                                                   g.splits, scale);
    return check_launch("conv_wgrad_reduce");
}

// ---- DCN site kernel (dcn_site.cuh): windows of x staged in shared memory; conv_offset optionally fused in front
size_t eb_dcn_site_offset_weight_bytes(int C) { return static_cast<size_t>(C / 32) * 9 * DS_WO_STAGE; }

int eb_dcn_site_pack_offset_weight(const float* wo, const float* bo, int C, int dg, void* wo_pack, float* bo_cols, void* stream) {
    if (!wo || !wo_pack || !bo_cols) return fail(EB_ERR_NULLPTR, "dcn_site_pack: null pointer");
    if (C < 64 || C % 64 || dg < 1 || dg * 27 > DS_OFF_N) return fail(EB_ERR_INVALID_SHAPE, "dcn_site_pack: C=%d dg=%d", C, dg);
    const long long groups = static_cast<long long>(C / 32) * 9 * 4 * DS_OFF_N;
    pack_offset_weight_kernel<<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        wo, bo, C, dg, DS_OFF_N, static_cast<__half*>(wo_pack), bo_cols);
    return check_launch("pack_offset_weight");
}

int eb_dcn_site(const void* x, int x_pix_stride, int x_ch_off, int N, int H, int W, int C, int dg,
                const float* offset, const float* mask, long long off_img_stride, long long mask_img_stride, int mask_logit,
                const void* feat, int f_pix_stride, int f_ch_off, const void* wo_pack, const float* bo_cols,
                const void* wpack, int BN, int n_tiles_n, const eb_epilogue_t* epi, float* absmean, void* stream) {
    const bool fused = feat != nullptr;
    if (!x || !wpack || (fused ? (!wo_pack || !bo_cols) : !offset)) return fail(EB_ERR_NULLPTR, "dcn_site: null pointer");
    if (N < 0 || H < 1 || W < 1 || C < 64 || C % 64 || dg < 1 || C % dg || ((C / dg) != 8 && (C / dg) % 16))
        return fail(EB_ERR_INVALID_SHAPE, "dcn_site: N=%d H=%d W=%d C=%d dg=%d (C/dg must be 8 or a multiple of 16)", N, H, W, C, dg);
    if (BN % 32 || BN < 32 || BN > 128 || n_tiles_n < 1 || BN * n_tiles_n > DC_MAX_COUT)
        return fail(EB_ERR_INVALID_SHAPE, "dcn_site: BN=%d n_tiles_n=%d", BN, n_tiles_n);
    if (!al16(x) || !al16(wpack) || x_pix_stride % 8 || x_ch_off % 8 || x_pix_stride < x_ch_off + C)
        return fail(EB_ERR_ALIGNMENT, "dcn_site: x view must be 16-byte aligned");
    if (fused && (dg * 27 > DS_OFF_N || !al16(feat) || !al16(wo_pack) || f_pix_stride % 8 || f_ch_off % 8 || f_pix_stride < f_ch_off + C))
        return fail(EB_ERR_UNSUPPORTED, "dcn_site: fused conv_offset needs dg*27 <= %d and a 16-byte aligned feature view", DS_OFF_N);
    eb_encode_tiled_fn enc = tensor_map_encoder();
    if (!enc) return fail(EB_ERR_UNSUPPORTED, "dcn_site: cuTensorMapEncodeTiled unavailable");
    if (N == 0) return EB_OK;
    DsParams PP;
    memset(&PP, 0, sizeof(PP));
    DcnParams& P = PP.d;
    P.x = static_cast<const __half*>(x); P.x_pix_stride = x_pix_stride; P.x_ch_off = x_ch_off;
    P.N = N; P.H = H; P.W = W; P.C = C; P.Ho = H; P.Wo = W;
    P.kh = 3; P.kw = 3; P.stride = 1; P.pad = 1; P.dil = 1; P.stride_w = 1; P.pad_w = 1; P.dil_w = 1;
    P.dg = dg; P.cpg = C / dg;
    P.x_wide = (x_pix_stride % 16 == 0 && x_ch_off % 16 == 0 && reinterpret_cast<uintptr_t>(x) % 32 == 0) ? 1 : 0;
    P.offset = offset; P.mask = mask;
    P.wpack = static_cast<const __half*>(wpack); P.BN = BN; P.n_tiles_n = n_tiles_n;
    if (int rc = fill_epi(epi, H, W, BN * n_tiles_n, &P.epi)) return rc;
    if (P.epi.out_mode != OUT_SAME) return fail(EB_ERR_UNSUPPORTED, "dcn_site: out_mode");
    const bool nchw = P.epi.out_nchw != nullptr;
    if (nchw && (P.epi.out16 || P.epi.out32 || P.epi.res16 || P.epi.res32)) return fail(EB_ERR_UNSUPPORTED, "dcn_site: NCHW output excludes other outputs");
    if (!nchw && (!P.epi.out16 || P.epi.out32 || P.epi.res32 || P.epi.res16)) return fail(EB_ERR_UNSUPPORTED, "dcn_site: NHWC fp16 output only");
    PP.off_img_stride = off_img_stride; PP.mask_img_stride = mask_img_stride; PP.mask_logit = mask_logit;
    PP.absmean = absmean;
    PP.f_ch_off = f_ch_off; PP.wo_pack = static_cast<const __half*>(wo_pack); PP.bo = bo_cols;
    {
        const cuuint64_t ps = static_cast<cuuint64_t>(x_pix_stride);
        const cuuint64_t dims[4] = {ps, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[3] = {ps * 2, static_cast<cuuint64_t>(W) * ps * 2, static_cast<cuuint64_t>(H) * W * ps * 2};
        const cuuint32_t box[4] = {64, DS_WW, DS_WH, 1};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult r = enc(&PP.tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(x), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "dcn_site: window tensor map failed (%d)", static_cast<int>(r));
    }
    PP.tmap_f = PP.tmap_x;
    if (fused) {
        const cuuint64_t ps = static_cast<cuuint64_t>(f_pix_stride);
        const cuuint64_t dims[5] = {8, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), ps / 8, static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[4] = {ps * 2, static_cast<cuuint64_t>(W) * ps * 2, 16, static_cast<cuuint64_t>(H) * W * ps * 2};
        const cuuint32_t box[5] = {8, DS_F_RP_X, DS_F_RP_Y, 4, 1};
        const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
        const CUresult r = enc(&PP.tmap_f, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(feat), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "dcn_site: feature tensor map failed (%d)", static_cast<int>(r));
    }
    const long long tiles = static_cast<long long>(N) * ((H + DC_TILE_H - 1) / DC_TILE_H) * ((W + DC_TILE_W - 1) / DC_TILE_W) * n_tiles_n;
    int grid = static_cast<int>(tiles < num_sms() ? tiles : num_sms());
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // clusters of two CTAs share one L2 read of every weight stage (811 KB of weights are re-streamed per 128-pixel tile)
    const char* mc_env = getenv("EDVR_B200_DCN_MC");
    PP.multicast = (grid >= 2 && !(mc_env && mc_env[0] == '0')) ? 1 : 0;
    if (PP.multicast) grid &= ~1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(DS_THREADS);
    cfg.dynamicSmemBytes = DS_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = PP.multicast ? 1 : 0;
    cudaError_t lerr = cudaSuccess;
    const bool two = P.cpg == 8;       // two deformable groups per 16-channel K-atom pair (EDVR-M: 64 channels, dg 8)
#define EB_LAUNCH_DS(OFF_, EK_)                                                                        \
    do {                                                                                               \
        if (two) {                                                                                     \
            if (int rc = set_smem(dcn_site_kernel<OFF_, EK_, true>, DS_SMEM_BYTES)) return rc;         \
            lerr = cudaLaunchKernelEx(&cfg, dcn_site_kernel<OFF_, EK_, true>, PP);                     \
        } else {                                                                                       \
            if (int rc = set_smem(dcn_site_kernel<OFF_, EK_, false>, DS_SMEM_BYTES)) return rc;        \
            lerr = cudaLaunchKernelEx(&cfg, dcn_site_kernel<OFF_, EK_, false>, PP);                    \
        }                                                                                              \
    } while (0)
    if (fused) { if (nchw) EB_LAUNCH_DS(DS_OFF_TMEM, EK_NCHW); else EB_LAUNCH_DS(DS_OFF_TMEM, EK_PLAIN); }
    else       { if (nchw) EB_LAUNCH_DS(DS_OFF_GLOBAL, EK_NCHW); else EB_LAUNCH_DS(DS_OFF_GLOBAL, EK_PLAIN); }
#undef EB_LAUNCH_DS
    if (lerr != cudaSuccess) return fail(EB_ERR_LAUNCH, "dcn_site: %s", cudaGetErrorString(lerr));
    return check_launch("dcn_site");
}

// ---- CTA-pair DCN site kernel (dcn_pair.cuh): conv_offset of the next half tile overlaps the gather of this one
int eb_dcn_pair_supported(int C, int dg, int BN, int n_tiles_n) {
    if (C < 64 || C % 64 || dg < 2 || dg % 2 || C % dg || (dg / 2) * 27 > DP_OFF_HALF) return 0;
    const int cpg = C / dg;
    if (cpg != 8 && cpg % 16) return 0;
    if (BN % 32 || BN < 32 || BN > 128 || n_tiles_n != 1) return 0;
    if (num_sms() < 2 || tensor_map_encoder() == nullptr) return 0;
    return 1;
}

size_t eb_dcn_pair_offset_weight_bytes(int C) { return static_cast<size_t>(4) * (C / 32) * 9 * DP_WO_TAP; }

int eb_dcn_pair_pack_offset_weight(const float* wo, const float* bo, int C, int dg, void* wo_pack, float* bo_cols, void* stream) {
    if (!wo || !wo_pack || !bo_cols) return fail(EB_ERR_NULLPTR, "dcn_pair_pack: null pointer");
    if (C < 64 || C % 64 || dg < 2 || dg % 2 || (dg / 2) * 27 > DP_OFF_HALF) return fail(EB_ERR_INVALID_SHAPE, "dcn_pair_pack: C=%d dg=%d", C, dg);
    const long long groups = 4ll * (C / 32) * 9 * 4 * DP_WO_ROWS;
    pack_offset_weight_pair_kernel<<<grid_1d(groups, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        wo, bo, C, dg, static_cast<__half*>(wo_pack), bo_cols);
    return check_launch("pack_offset_weight_pair");
}

// Role timing counters of dcn_pair_kernel (library built with -DDP_PROF; otherwise reads zeros): copies the 32 counters to
// `host` (synchronises the device) and clears them.
static unsigned long long* dp_prof_buffer() {
    static unsigned long long* buf = nullptr;
    if (!buf && cudaMalloc(&buf, 32 * sizeof(unsigned long long)) == cudaSuccess) cudaMemset(buf, 0, 32 * sizeof(unsigned long long));
    return buf;
}
int eb_dcn_pair_prof_read(unsigned long long* host) {
    if (!host) return fail(EB_ERR_NULLPTR, "dcn_pair_prof_read: null pointer");
    unsigned long long* buf = dp_prof_buffer();
    if (!buf) return fail(EB_ERR_LAUNCH, "dcn_pair_prof_read: no buffer");
    if (cudaMemcpy(host, buf, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return fail(EB_ERR_LAUNCH, "dcn_pair_prof_read: copy");
    cudaMemset(buf, 0, 32 * sizeof(unsigned long long));
    return EB_OK;
}

int eb_dcn_site_pair(const void* x, int x_pix_stride, int x_ch_off, int N, int H, int W, int C, int dg,
                     const void* feat, int f_pix_stride, int f_ch_off, const void* wo_pack, const float* bo_cols,
                     const void* wpair, int BN, const eb_epilogue_t* epi, float* absmean, void* stream) {
    if (!x || !feat || !wo_pack || !bo_cols || !wpair) return fail(EB_ERR_NULLPTR, "dcn_site_pair: null pointer");
    if (N < 0 || H < 1 || W < 1) return fail(EB_ERR_INVALID_SHAPE, "dcn_site_pair: N=%d H=%d W=%d", N, H, W);
    if (!eb_dcn_pair_supported(C, dg, BN, 1))
        return fail(EB_ERR_UNSUPPORTED, "dcn_site_pair: C=%d dg=%d BN=%d (see eb_dcn_pair_supported)", C, dg, BN);
    if (!al16(x) || !al16(wpair) || x_pix_stride % 8 || x_ch_off % 8 || x_pix_stride < x_ch_off + C)
        return fail(EB_ERR_ALIGNMENT, "dcn_site_pair: x view must be 16-byte aligned");
    if (!al16(feat) || !al16(wo_pack) || f_pix_stride % 8 || f_ch_off % 8 || f_pix_stride < f_ch_off + C)
        return fail(EB_ERR_ALIGNMENT, "dcn_site_pair: feature view must be 16-byte aligned");
    eb_encode_tiled_fn enc = tensor_map_encoder();
    if (N == 0) return EB_OK;
    DpParams PP;
    memset(&PP, 0, sizeof(PP));
    DcnParams& P = PP.d;
    P.x = static_cast<const __half*>(x); P.x_pix_stride = x_pix_stride; P.x_ch_off = x_ch_off;
    P.N = N; P.H = H; P.W = W; P.C = C; P.Ho = H; P.Wo = W;
    P.kh = 3; P.kw = 3; P.stride = 1; P.pad = 1; P.dil = 1; P.stride_w = 1; P.pad_w = 1; P.dil_w = 1;
    P.dg = dg; P.cpg = C / dg;
    P.x_wide = (x_pix_stride % 16 == 0 && x_ch_off % 16 == 0 && reinterpret_cast<uintptr_t>(x) % 32 == 0) ? 1 : 0;
    P.wpack = static_cast<const __half*>(wpair); P.BN = BN; P.n_tiles_n = 1;
    if (int rc = fill_epi(epi, H, W, BN, &P.epi)) return rc;
    if (P.epi.out_mode != OUT_SAME) return fail(EB_ERR_UNSUPPORTED, "dcn_site_pair: out_mode");
    const bool nchw = P.epi.out_nchw != nullptr;
    if (nchw && (P.epi.out16 || P.epi.out32 || P.epi.res16 || P.epi.res32)) return fail(EB_ERR_UNSUPPORTED, "dcn_site_pair: NCHW output excludes other outputs");
    if (!nchw && (!P.epi.out16 || P.epi.out32 || P.epi.res32 || P.epi.res16)) return fail(EB_ERR_UNSUPPORTED, "dcn_site_pair: NHWC fp16 output only");
    PP.absmean = absmean;
    PP.f_ch_off = f_ch_off; PP.wo_pack = static_cast<const __half*>(wo_pack); PP.bo = bo_cols;
    { const char* e = getenv("EDVR_B200_DP_DBG"); PP.dbg = e ? atoi(e) : 0; }      // profiling ablations, results are wrong when set
    { const char* e = getenv("EDVR_B200_DP_HINT_CRIT"); PP.hint_crit = e ? atoi(e) : 0; }
    { const char* e = getenv("EDVR_B200_DP_HINT_IDLE"); PP.hint_idle = e ? atoi(e) : 2000; }
    { const char* e = getenv("EDVR_B200_DP_HINT_GATHER"); PP.hint_gather = e ? atoi(e) : 0; }
#ifdef DP_PROF
    PP.prof = dp_prof_buffer();
#endif
    {
        const cuuint64_t ps = static_cast<cuuint64_t>(x_pix_stride);
        const cuuint64_t dims[4] = {ps, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[3] = {ps * 2, static_cast<cuuint64_t>(W) * ps * 2, static_cast<cuuint64_t>(H) * W * ps * 2};
        const cuuint32_t box[4] = {32, DP_WW, DP_WH, 1};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult r = enc(&PP.tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(x), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "dcn_site_pair: window tensor map failed (%d)", static_cast<int>(r));
    }
    {
        const cuuint64_t ps = static_cast<cuuint64_t>(f_pix_stride);
        const cuuint64_t dims[5] = {8, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), ps / 8, static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[4] = {ps * 2, static_cast<cuuint64_t>(W) * ps * 2, 16, static_cast<cuuint64_t>(H) * W * ps * 2};
        const cuuint32_t box[5] = {8, DS_F_RP_X, DS_F_RP_Y, 4, 1};
        const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
        const CUresult r = enc(&PP.tmap_f, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(feat), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "dcn_site_pair: feature tensor map failed (%d)", static_cast<int>(r));
    }
    {
        // packed weight arrays as rows of 256 fp16 (512 B); one box = one pipeline stage of one CTA, landing as a linear copy
        const cuuint32_t estr[2] = {1, 1};
        const cuuint64_t strides[1] = {512};
        const cuuint64_t dims_w[2] = {256, static_cast<cuuint64_t>(2) * (C / 32) * 9 * (BN / 16)};
        const cuuint32_t box_w[2] = {256, static_cast<cuuint32_t>(BN / 16)};
        CUresult r = enc(&PP.tmap_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(wpair), dims_w, strides, box_w, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "dcn_site_pair: weight tensor map failed (%d)", static_cast<int>(r));
        const cuuint64_t dims_o[2] = {256, static_cast<cuuint64_t>(4) * (C / 32) * 3 * (DP_WO_STAGE / 512)};
        const cuuint32_t box_o[2] = {256, DP_WO_STAGE / 512};
        r = enc(&PP.tmap_wo, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(wo_pack), dims_o, strides, box_o, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(EB_ERR_LAUNCH, "dcn_site_pair: offset weight tensor map failed (%d)", static_cast<int>(r));
    }
    const long long tiles = static_cast<long long>(N) * ((H + DC_TILE_H - 1) / DC_TILE_H) * ((W + DC_TILE_W - 1) / DC_TILE_W);
    const long long npairs = (tiles + 1) / 2;
    const int max_clusters = num_sms() / 2;
    const int nclusters = static_cast<int>(npairs < max_clusters ? npairs : max_clusters);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * nclusters);
    cfg.blockDim = dim3(DP_THREADS);
    cfg.dynamicSmemBytes = DP_SMEM_BYTES;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;      // see pdl_wait() in dcn_pair.cuh
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = getenv("EDVR_B200_NO_PDL") ? 1 : 2;
    cudaError_t lerr = cudaSuccess;
    const bool two = P.cpg == 8;
#define EB_LAUNCH_DP(EK_)                                                                          \
    do {                                                                                           \
        if (two) {                                                                                 \
            if (int rc = set_smem(dcn_pair_kernel<EK_, true>, DP_SMEM_BYTES)) return rc;           \
            lerr = cudaLaunchKernelEx(&cfg, dcn_pair_kernel<EK_, true>, PP);                       \
        } else {                                                                                   \
            if (int rc = set_smem(dcn_pair_kernel<EK_, false>, DP_SMEM_BYTES)) return rc;          \
            lerr = cudaLaunchKernelEx(&cfg, dcn_pair_kernel<EK_, false>, PP);                      \
        }                                                                                          \
    } while (0)
    if (nchw) EB_LAUNCH_DP(EK_NCHW); else EB_LAUNCH_DP(EK_PLAIN);
#undef EB_LAUNCH_DP
    if (lerr != cudaSuccess) return fail(EB_ERR_LAUNCH, "dcn_site_pair: %s", cudaGetErrorString(lerr));
    return check_launch("dcn_site_pair");
}

// ---- reference-layout operator -----------------------------------------------------------
static inline size_t up256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }
static inline int cout_tiles(int Cout, int* BN) {
    int bn = Cout >= 128 ? 128 : ((Cout + 31) / 32) * 32;
    *BN = bn;
    return (Cout + bn - 1) / bn;
}

size_t eb_mdcn_forward_workspace(int N, int C, int H, int W, int Cout, int kh, int kw) {
    int BN;
    const int nt = cout_tiles(Cout, &BN);
    return up256(static_cast<size_t>(N) * H * W * C * 2) + up256(eb_packed_weight_bytes(C, kh * kw, BN, nt)) +
           up256(static_cast<size_t>(BN) * nt * 4);
}

namespace {
struct Geo2 { int sh, sw, ph, pw, dh, dw; };

// Shared implementation of the reference-layout forward: mask == NULL and bias == NULL give DCNv1.
int dcn_forward_impl(const char* who, const float* x, const float* offset, const float* mask, const float* weight,
                     const float* bias, float* out, int N, int C, int H, int W, int Cout, int kh, int kw, Geo2 g,
                     int groups, int dg, void* workspace, size_t workspace_bytes, void* stream, bool need_mask,
                     const __half* x_half = nullptr) {      // x_half: the input as an fp16 NCHW tensor instead of x
    if (N == 0 && C > 0 && H > 0 && W > 0 && Cout > 0) return EB_OK;   // empty batch: nothing to do, pointers may be NULL
    if ((!x && !x_half) || !offset || (need_mask && !mask) || !weight || !out) return fail(EB_ERR_NULLPTR, "%s: null pointer", who);
    if (N < 0 || C < 1 || H < 1 || W < 1 || Cout < 1 || kh < 1 || kw < 1 || g.sh < 1 || g.sw < 1 || g.ph < 0 || g.pw < 0 ||
        g.dh < 1 || g.dw < 1 || groups < 1 || dg < 1 || C % dg || C % groups || Cout % groups)
        return fail(EB_ERR_INVALID_SHAPE, "%s: invalid shape", who);
    if (groups != 1) return fail(EB_ERR_UNSUPPORTED, "%s: groups=%d (only 1; EDVR uses 1)", who, groups);
    if (C % 64 || (C / dg) % 8) return fail(EB_ERR_UNSUPPORTED, "%s: C=%d dg=%d (C %% 64 == 0, (C/dg) %% 8 == 0)", who, C, dg);
    if (Cout > DC_MAX_COUT) return fail(EB_ERR_UNSUPPORTED, "%s: Cout=%d > %d", who, Cout, DC_MAX_COUT);
    const int Ho = (H + 2 * g.ph - (g.dh * (kh - 1) + 1)) / g.sh + 1;
    const int Wo = (W + 2 * g.pw - (g.dw * (kw - 1) + 1)) / g.sw + 1;
    if (Ho < 1 || Wo < 1) return fail(EB_ERR_INVALID_SHAPE, "%s: empty output", who);
    const size_t need = eb_mdcn_forward_workspace(N, C, H, W, Cout, kh, kw);
    if (workspace_bytes < need || !workspace) return fail(EB_ERR_WORKSPACE, "%s: workspace %zu < %zu", who, workspace_bytes, need);
    if (!al16(workspace)) return fail(EB_ERR_ALIGNMENT, "%s: workspace must be 16-byte aligned", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int BN;
    const int nt = cout_tiles(Cout, &BN);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    __half* x16 = reinterpret_cast<__half*>(ws);
    ws += up256(static_cast<size_t>(N) * H * W * C * 2);
    __half* wpack = reinterpret_cast<__half*>(ws);
    ws += up256(eb_packed_weight_bytes(C, kh * kw, BN, nt));
    float* bpack = reinterpret_cast<float*>(ws);
    {
        dim3 grid((H * W + 31) / 32, (C + 31) / 32, N), block(32, 8);
        if (x_half) nchw_f16_to_nhwc_f16_kernel<<<grid, block, 0, st>>>(x_half, x16, C, H * W);
        else nchw_f32_to_nhwc_f16_kernel<<<grid, block, 0, st>>>(x, x16, C, H * W, C, 0);
        if (int rc = check_launch("nchw_to_nhwc")) return rc;
    }
    if (int rc = eb_pack_weight(weight, Cout, C, kh * kw, BN, nt, wpack, stream)) return rc;
    pack_bias_kernel<<<(BN * nt + 127) / 128, 128, 0, st>>>(bias, Cout, BN * nt, bpack);
    if (int rc = check_launch("pack_bias")) return rc;

    DcnParams P;
    memset(&P, 0, sizeof(P));
    P.x = x16; P.x_pix_stride = C; P.x_ch_off = 0;
    P.N = N; P.H = H; P.W = W; P.C = C; P.Ho = Ho; P.Wo = Wo;
    P.kh = kh; P.kw = kw; P.stride = g.sh; P.pad = g.ph; P.dil = g.dh; P.stride_w = g.sw; P.pad_w = g.pw; P.dil_w = g.dw;
    P.dg = dg; P.cpg = C / dg;
    P.x_wide = (P.cpg % 16 == 0 && reinterpret_cast<uintptr_t>(x16) % 32 == 0) ? 1 : 0;   // pixel stride C % 64 == 0, offset 0
    P.offset = offset; P.mask = mask;
    P.wpack = wpack; P.BN = BN; P.n_tiles_n = nt;
    P.epi.bias = bias ? bpack : nullptr; P.epi.act = ACT_NONE; P.epi.H = Ho; P.epi.W = Wo;
    P.epi.out_nchw = out; P.epi.nchw_C = Cout; P.epi.out_mode = OUT_SAME;
    const long long tiles = static_cast<long long>(N) * ((Ho + DC_TILE_H - 1) / DC_TILE_H) * ((Wo + DC_TILE_W - 1) / DC_TILE_W) * nt;
    const int grid = static_cast<int>(tiles < num_sms() ? tiles : num_sms());
    // keep the rest of the 228 KB for L1: the nine taps of a chunk re-read the same slab of x
    static const int carve = (DC_SMEM_BYTES + 1024) * 100 / (228 * 1024) + 1;
    cudaFuncSetAttribute(dcn_fused_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    if (int rc = set_smem(dcn_fused_kernel, DC_SMEM_BYTES)) return rc;
    dcn_fused_kernel<<<grid, DC_THREADS, DC_SMEM_BYTES, st>>>(P);
    return check_launch("dcn_fused");
}
}  // namespace

int eb_mdcn_forward(const float* x, const float* offset, const float* mask, const float* weight,
                    const float* bias, float* out, int N, int C, int H, int W, int Cout, int kh, int kw,
                    int stride, int pad, int dil, int groups, int dg, void* workspace,
                    size_t workspace_bytes, void* stream) {
    return dcn_forward_impl("mdcn_forward", x, offset, mask, weight, bias, out, N, C, H, W, Cout, kh, kw,
                            Geo2{stride, stride, pad, pad, dil, dil}, groups, dg, workspace, workspace_bytes, stream, true);
}

/* Half-precision operator entry: what the reference's AT_DISPATCH_FLOATING_TYPES_AND_HALF instantiation answers for
 * at::Half tensors (deform_conv_cuda_kernel.cu:781-800, deform_conv_cuda.cpp:490-569).  All tensors fp16 in the reference
 * layouts; the arithmetic is the library's (fp16 tensor-core operands - the input is used as given, no re-rounding -, fp32
 * offsets / masks / accumulation), the result is rounded to fp16 once. */
size_t eb_mdcn_forward_f16_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int dg) {
    // fp32 copies of offset, mask, weight, bias and the fp32 result, sized for outputs of at most H x W pixels (checked by
    // eb_mdcn_forward_f16: the usual "same" or strided geometries)
    const size_t hw = static_cast<size_t>(H) * W, k = static_cast<size_t>(kh) * kw;
    return eb_mdcn_forward_workspace(N, C, H, W, Cout, kh, kw) + up256(N * dg * 2 * k * hw * 4) + up256(N * dg * k * hw * 4) +
           up256(static_cast<size_t>(Cout) * C * k * 4) + up256(static_cast<size_t>(Cout) * 4) + up256(N * Cout * hw * 4);
}

int eb_mdcn_forward_f16(const void* x, const void* offset, const void* mask, const void* weight, const void* bias, void* out,
                        int N, int C, int H, int W, int Cout, int kh, int kw, int stride, int pad, int dil, int groups, int dg,
                        void* workspace, size_t workspace_bytes, void* stream) {
    if (N == 0 && C > 0 && H > 0 && W > 0 && Cout > 0) return EB_OK;
    if (!x || !offset || !mask || !weight || !out) return fail(EB_ERR_NULLPTR, "mdcn_forward_f16: null pointer");
    if (N < 0 || C < 1 || H < 1 || W < 1 || Cout < 1 || kh < 1 || kw < 1 || stride < 1 || pad < 0 || dil < 1 || dg < 1)
        return fail(EB_ERR_INVALID_SHAPE, "mdcn_forward_f16: invalid shape");
    const int Ho = (H + 2 * pad - (dil * (kh - 1) + 1)) / stride + 1, Wo = (W + 2 * pad - (dil * (kw - 1) + 1)) / stride + 1;
    if (Ho < 1 || Wo < 1) return fail(EB_ERR_INVALID_SHAPE, "mdcn_forward_f16: empty output");
    if (static_cast<long long>(Ho) * Wo > static_cast<long long>(H) * W)
        return fail(EB_ERR_UNSUPPORTED, "mdcn_forward_f16: output larger than the input (padding beyond the kernel reach)");
    const size_t need = eb_mdcn_forward_f16_workspace(N, C, H, W, Cout, kh, kw, dg);
    if (!workspace || workspace_bytes < need) return fail(EB_ERR_WORKSPACE, "mdcn_forward_f16: workspace %zu < %zu", workspace_bytes, need);
    if (!al16(workspace)) return fail(EB_ERR_ALIGNMENT, "mdcn_forward_f16: workspace must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    const size_t inner = eb_mdcn_forward_workspace(N, C, H, W, Cout, kh, kw);
    uint8_t* cur = ws + inner;
    auto take = [&](size_t elems) { float* p = reinterpret_cast<float*>(cur); cur += up256(elems * 4); return p; };
    const long long n_off = static_cast<long long>(N) * dg * 2 * kh * kw * Ho * Wo, n_mask = n_off / 2;
    const long long n_w = static_cast<long long>(Cout) * (C / (groups > 0 ? groups : 1)) * kh * kw, n_out = static_cast<long long>(N) * Cout * Ho * Wo;
    float* off32 = take(static_cast<size_t>(N) * dg * 2 * kh * kw * H * W);
    float* mask32 = take(static_cast<size_t>(N) * dg * kh * kw * H * W);
    float* w32 = take(static_cast<size_t>(Cout) * C * kh * kw);
    float* b32 = take(Cout);
    float* out32 = take(static_cast<size_t>(N) * Cout * H * W);
    auto to_f32 = [&](const void* src, float* dst, long long n) {
        half_to_float_kernel<<<grid_1d(n, 256), 256, 0, st>>>(static_cast<const __half*>(src), dst, n);
    };
    to_f32(offset, off32, n_off);
    to_f32(mask, mask32, n_mask);
    to_f32(weight, w32, n_w);
    if (bias) to_f32(bias, b32, Cout);
    if (int rc = check_launch("half_to_float")) return rc;
    if (int rc = dcn_forward_impl("mdcn_forward_f16", nullptr, off32, mask32, w32, bias ? b32 : nullptr, out32, N, C, H, W, Cout, kh, kw,
                                  Geo2{stride, stride, pad, pad, dil, dil}, groups, dg, ws, inner, stream, true,
                                  static_cast<const __half*>(x)))
        return rc;
    float_to_half_kernel<<<grid_1d(n_out, 256), 256, 0, st>>>(out32, static_cast<__half*>(out), n_out);
    return check_launch("float_to_half");
}

/* DCNv1: deform_conv_forward of the reference extension (deform_conv_ext.cpp:51-67, deform_conv_cuda.cpp:152-237) */
int eb_dcn1_forward(const float* x, const float* offset, const float* weight, float* out, int N, int C, int H, int W,
                    int Cout, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                    int groups, int dg, void* workspace, size_t workspace_bytes, void* stream) {
    return dcn_forward_impl("dcn1_forward", x, offset, nullptr, weight, nullptr, out, N, C, H, W, Cout, kh, kw,
                            Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, groups, dg, workspace, workspace_bytes,
                            stream, false);
}

namespace {
struct BwdWs {
    size_t x16, go16, wT, gcol16, gx32, colT, goT, total;
    int Cout64, BN, mt;
    long long P, Ppad;
};
BwdWs bwd_ws(int N, int C, int H, int W, int Cout, int K, int Ho, int Wo) {
    BwdWs w;
    w.Cout64 = ((Cout + 63) / 64) * 64;
    w.BN = (C % 128 == 0) ? 128 : 64;
    w.mt = (Cout + 127) / 128;
    w.P = static_cast<long long>(N) * Ho * Wo;
    w.Ppad = ((w.P + 63) / 64) * 64;
    size_t o = 0;
    w.x16 = o;    o += up256(static_cast<size_t>(N) * H * W * C * 2);
    w.go16 = o;   o += up256(static_cast<size_t>(w.P) * w.Cout64 * 2);
    w.wT = o;     o += up256(static_cast<size_t>(K) * C * w.Cout64 * 2);
    w.gcol16 = o; o += up256(static_cast<size_t>(w.P) * K * C * 2);
    w.gx32 = o;   o += up256(static_cast<size_t>(N) * H * W * C * 4);
    w.colT = o;   o += up256(static_cast<size_t>(K) * C * w.Ppad * 2);
    w.goT = o;    o += up256(static_cast<size_t>(w.mt) * 128 * w.Ppad * 2);
    w.total = o;
    return w;
}
}  // namespace

static size_t bwd_workspace2(int N, int C, int H, int W, int Cout, int kh, int kw, Geo2 g) {
    const int Ho = (H + 2 * g.ph - (g.dh * (kh - 1) + 1)) / g.sh + 1;
    const int Wo = (W + 2 * g.pw - (g.dw * (kw - 1) + 1)) / g.sw + 1;
    if (Ho < 1 || Wo < 1 || N < 1) return 256;
    return bwd_ws(N, C, H, W, Cout, kh * kw, Ho, Wo).total;
}

size_t eb_mdcn_backward_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride,
                                  int pad, int dil) {
    return bwd_workspace2(N, C, H, W, Cout, kh, kw, Geo2{stride, stride, pad, pad, dil, dil});
}

size_t eb_dcn1_backward_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h, int stride_w,
                                  int pad_h, int pad_w, int dil_h, int dil_w) {
    return bwd_workspace2(N, C, H, W, Cout, kh, kw, Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w});
}

namespace {
// Shared backward: `want_input` -> grad_x, grad_offset (and grad_mask when mask != NULL); `want_param` ->
// grad_weight += scale * (...), grad_bias += (...).  mask == NULL gives DCNv1.
int dcn_backward_impl(const char* who, const float* x, const float* offset, const float* mask, const float* weight,
                      const float* grad_out, float* grad_x, float* grad_offset, float* grad_mask, float* grad_weight,
                      float* grad_bias, float scale, bool want_input, bool want_param, int N, int C, int H, int W,
                      int Cout, int kh, int kw, Geo2 g, int groups, int dg, void* workspace, size_t workspace_bytes,
                      void* stream) {
    if (N == 0 && C > 0 && H > 0 && W > 0 && Cout > 0) return EB_OK;   // empty batch
    if (!x || !offset || !grad_out || (want_input && (!weight || !grad_x || !grad_offset)) || (want_param && !grad_weight))
        return fail(EB_ERR_NULLPTR, "%s: null pointer", who);
    if (N < 0 || C < 1 || H < 1 || W < 1 || Cout < 1 || kh < 1 || kw < 1 || g.sh < 1 || g.sw < 1 || g.ph < 0 || g.pw < 0 ||
        g.dh < 1 || g.dw < 1 || groups < 1 || dg < 1 || C % dg || C % groups || Cout % groups)
        return fail(EB_ERR_INVALID_SHAPE, "%s: invalid shape", who);
    if (groups != 1) return fail(EB_ERR_UNSUPPORTED, "%s: groups=%d (only 1; EDVR uses 1)", who, groups);
    if (C % 64 || (C / dg) % 8) return fail(EB_ERR_UNSUPPORTED, "%s: C=%d dg=%d (C %% 64 == 0, (C/dg) %% 8 == 0)", who, C, dg);
    const int Ho = (H + 2 * g.ph - (g.dh * (kh - 1) + 1)) / g.sh + 1;
    const int Wo = (W + 2 * g.pw - (g.dw * (kw - 1) + 1)) / g.sw + 1;
    if (Ho < 1 || Wo < 1) return fail(EB_ERR_INVALID_SHAPE, "%s: empty output", who);
    const int K = kh * kw;
    const BwdWs ws = bwd_ws(N, C, H, W, Cout, K, Ho, Wo);
    if (!workspace || workspace_bytes < ws.total)
        return fail(EB_ERR_WORKSPACE, "%s: workspace %zu < %zu", who, workspace_bytes, ws.total);
    if (!al16(workspace)) return fail(EB_ERR_ALIGNMENT, "%s: workspace must be 16-byte aligned", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* base = static_cast<uint8_t*>(workspace);
    __half* x16 = reinterpret_cast<__half*>(base + ws.x16);
    __half* go16 = reinterpret_cast<__half*>(base + ws.go16);
    __half* wT = reinterpret_cast<__half*>(base + ws.wT);
    __half* gcol16 = reinterpret_cast<__half*>(base + ws.gcol16);
    float* gx32 = reinterpret_cast<float*>(base + ws.gx32);
    __half* colT = reinterpret_cast<__half*>(base + ws.colT);
    __half* goT = reinterpret_cast<__half*>(base + ws.goT);
    DcnBwdGeom G{N, C, H, W, Cout, kh, kw, g.sh, g.ph, g.dh, dg, Ho, Wo, g.sw, g.pw, g.dw};
    const int HWo = Ho * Wo;

    {   // layouts
        dim3 block(32, 8);
        nchw_f32_to_nhwc_f16_kernel<<<dim3((H * W + 31) / 32, (C + 31) / 32, N), block, 0, st>>>(x, x16, C, H * W, C, 0);
        if (int rc = check_launch("bwd layouts")) return rc;
    }
    if (want_input) {
        // stage 1: gcol = W^T . gO as a 1x1 conv with K*C output channels
        dim3 block(32, 8);
        if (ws.Cout64 != Cout) cudaMemsetAsync(go16, 0, static_cast<size_t>(ws.P) * ws.Cout64 * 2, st);
        nchw_f32_to_nhwc_f16_kernel<<<dim3((HWo + 31) / 32, (Cout + 31) / 32, N), block, 0, st>>>(grad_out, go16, Cout, HWo, ws.Cout64, 0);
        const long long groups16 = static_cast<long long>(K) * C * (ws.Cout64 / 8);
        pack_wT_kernel<<<grid_1d(groups16, 256), 256, 0, st>>>(weight, Cout, C, K, ws.Cout64, ws.BN, wT);
        ConvParams P;
        memset(&P, 0, sizeof(P));
        P.src[0].ptr = go16; P.src[0].C = ws.Cout64; P.src[0].pix_stride = ws.Cout64; P.src[0].ch_off = 0;
        P.src[0].div = 1; P.src[0].mul = 1; P.src[0].keep = 0; P.src[0].add = 0;
        P.nsrc = 1; P.N = N; P.H = Ho; P.W = Wo; P.taps = 1; P.BN = ws.BN; P.n_tiles_n = K * C / ws.BN;
        P.wpack = wT;
        P.epi.act = ACT_NONE; P.epi.H = Ho; P.epi.W = Wo; P.epi.out16 = gcol16; P.epi.out16_pix_stride = K * C;
        P.epi.out_mode = OUT_SAME;
        if (int rc = launch_conv(P, st)) return rc;
        // stage 2: grad_offset, grad_mask, grad_input
        cudaMemsetAsync(gx32, 0, static_cast<size_t>(N) * H * W * C * 4, st);
        const long long items = static_cast<long long>(N) * dg * K * HWo;
        dcn_bwd_coord_scatter_kernel<<<grid_1d(items, 256), 256, 0, st>>>(G, x16, offset, mask, gcol16, gx32, grad_offset,
                                                                          mask ? grad_mask : nullptr);
        nhwc_f32_to_nchw_f32_kernel<<<dim3((H * W + 31) / 32, (C + 31) / 32, N), dim3(32, 8), 0, st>>>(gx32, grad_x, C, H * W);
        if (int rc = check_launch("bwd coord/scatter")) return rc;
    }
    if (want_param) {
        // stage 3: grad_weight (+= over the batch), grad_bias
        cudaMemsetAsync(goT, 0, static_cast<size_t>(ws.mt) * 128 * ws.Ppad * 2, st);
        if (ws.Ppad != ws.P) cudaMemsetAsync(colT, 0, static_cast<size_t>(K) * C * ws.Ppad * 2, st);
        dcn_bwd_goT_kernel<<<grid_1d(static_cast<long long>(N) * Cout * HWo, 256), 256, 0, st>>>(grad_out, goT, N, Cout, HWo, ws.Ppad);
        dcn_bwd_colT_kernel<<<grid_1d(static_cast<long long>(N) * (C / 8) * K * HWo, 256), 256, 0, st>>>(G, x16, offset, mask, colT, ws.Ppad);
        const int ntn = K * C / ws.BN;
        const long long steps = ws.Ppad / 64;
        long long want = (2LL * num_sms() + ntn * ws.mt - 1) / (ntn * ws.mt);   // ~2 waves of CTAs
        if (want < 1) want = 1;
        if (want > steps) want = steps;
        const int sps = static_cast<int>((steps + want - 1) / want);
        const int splits = static_cast<int>((steps + sps - 1) / sps);
        if (int rc = set_smem(dcn_bwd_wgrad_kernel, WG_SMEM_BYTES)) return rc;
        dcn_bwd_wgrad_kernel<<<dim3(ntn, ws.mt, splits), 128, WG_SMEM_BYTES, st>>>(goT, colT, grad_weight, Cout, C, K, ws.Ppad, ws.BN, sps, scale);
        if (grad_bias) dcn_bwd_bias_kernel<<<Cout, 256, 0, st>>>(grad_out, grad_bias, N, Cout, HWo);
        if (int rc = check_launch("bwd wgrad")) return rc;
    }
    return EB_OK;
}
}  // namespace

int eb_mdcn_backward(const float* x, const float* offset, const float* mask, const float* weight,
                     const float* grad_out, float* grad_x, float* grad_offset, float* grad_mask,
                     float* grad_weight, float* grad_bias, int N, int C, int H, int W, int Cout, int kh,
                     int kw, int stride, int pad, int dil, int groups, int dg, void* workspace,
                     size_t workspace_bytes, void* stream) {
    if (!(N == 0) && (!mask || !grad_mask)) return fail(EB_ERR_NULLPTR, "mdcn_backward: null pointer");
    return dcn_backward_impl("mdcn_backward", x, offset, mask, weight, grad_out, grad_x, grad_offset, grad_mask, grad_weight,
                             grad_bias, 1.0f, true, true, N, C, H, W, Cout, kh, kw, Geo2{stride, stride, pad, pad, dil, dil},
                             groups, dg, workspace, workspace_bytes, stream);
}

/* DCNv1: deform_conv_backward_input (deform_conv_ext.cpp:69-86, deform_conv_cuda.cpp:239-351): grad_x, grad_offset */
int eb_dcn1_backward_input(const float* x, const float* offset, const float* weight, const float* grad_out, float* grad_x,
                           float* grad_offset, int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h,
                           int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int groups, int dg, void* workspace,
                           size_t workspace_bytes, void* stream) {
    return dcn_backward_impl("dcn1_backward_input", x, offset, nullptr, weight, grad_out, grad_x, grad_offset, nullptr, nullptr,
                             nullptr, 1.0f, true, false, N, C, H, W, Cout, kh, kw,
                             Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, groups, dg, workspace, workspace_bytes, stream);
}

/* DCNv1: deform_conv_backward_parameters (deform_conv_ext.cpp:88-104, deform_conv_cuda.cpp:353-488): grad_weight += scale * dW */
int eb_dcn1_backward_parameters(const float* x, const float* offset, const float* grad_out, float* grad_weight, float scale,
                                int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h, int stride_w, int pad_h,
                                int pad_w, int dil_h, int dil_w, int groups, int dg, void* workspace, size_t workspace_bytes,
                                void* stream) {
    return dcn_backward_impl("dcn1_backward_parameters", x, offset, nullptr, nullptr, grad_out, nullptr, nullptr, nullptr,
                             grad_weight, nullptr, scale, false, true, N, C, H, W, Cout, kh, kw,
                             Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, groups, dg, workspace, workspace_bytes, stream);
}

// ---- fp64 reference-layout operator (dcn_f64.cuh) ---------------------------------------------------------------------
namespace {
constexpr int F64_MAX_Z = 65535;                                   // gridDim.z: images per launch
constexpr size_t F64_GCOL_BYTES = static_cast<size_t>(256) << 20;  // gcol staging target (at least one image)

// Argument checks shared by the fp64 entries: the statuses of the fp32 twins, without their C % 64 and Cout limits.
int f64_check(const char* who, bool ptrs_ok, int N, int C, int H, int W, int Cout, int kh, int kw, Geo2 g, int groups, int dg,
              F64Geom* G) {
    if (!ptrs_ok) return fail(EB_ERR_NULLPTR, "%s: null pointer", who);
    if (N < 0 || C < 1 || H < 1 || W < 1 || Cout < 1 || kh < 1 || kw < 1 || g.sh < 1 || g.sw < 1 || g.ph < 0 || g.pw < 0 ||
        g.dh < 1 || g.dw < 1 || groups < 1 || dg < 1 || C % dg || C % groups || Cout % groups)
        return fail(EB_ERR_INVALID_SHAPE, "%s: invalid shape", who);
    if (groups != 1) return fail(EB_ERR_UNSUPPORTED, "%s: groups=%d (only 1; compose weight groups above the ABI)", who, groups);
    const int Ho = (H + 2 * g.ph - (g.dh * (kh - 1) + 1)) / g.sh + 1;
    const int Wo = (W + 2 * g.pw - (g.dw * (kw - 1) + 1)) / g.sw + 1;
    if (Ho < 1 || Wo < 1) return fail(EB_ERR_INVALID_SHAPE, "%s: empty output", who);
    if (static_cast<long long>(N) * Ho * Wo > 0x7fffffffLL || static_cast<long long>(C) * kh * kw > 0x7fffffffLL)
        return fail(EB_ERR_UNSUPPORTED, "%s: more than 2^31 output pixels or C*kh*kw", who);
    // the GEMM grids put C*kh*kw (gcol, wgrad) and Cout (forward) tiles on gridDim.y
    if ((static_cast<long long>(C) * kh * kw + F64_BN - 1) / F64_BN > F64_MAX_Z || (Cout + F64_BN - 1) / F64_BN > F64_MAX_Z)
        return fail(EB_ERR_UNSUPPORTED, "%s: C*kh*kw or Cout above %d", who, F64_MAX_Z * F64_BN);
    *G = F64Geom{N, C, H, W, Cout, kh, kw, g.sh, g.sw, g.ph, g.pw, g.dh, g.dw, dg, Ho, Wo};
    return EB_OK;
}

int f64_forward_impl(const char* who, const double* x, const double* offset, const double* mask, const double* weight,
                     const double* bias, double* out, int N, int C, int H, int W, int Cout, int kh, int kw, Geo2 g, int groups,
                     int dg, void* stream, bool need_mask) {
    if (N == 0 && C > 0 && H > 0 && W > 0 && Cout > 0) return EB_OK;
    F64Geom G;
    if (int rc = f64_check(who, x && offset && (mask || !need_mask) && weight && out, N, C, H, W, Cout, kh, kw, g, groups, dg, &G))
        return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    F64FwdOp op;
    op.G = G; op.x = x; op.offset = offset; op.mask = mask; op.weight = weight; op.bias = bias; op.out = out;
    op.M = G.Ho * G.Wo; op.N = Cout;
    for (int n0 = 0; n0 < N; n0 += F64_MAX_Z) {
        op.n_first = n0;
        const dim3 grid((op.M + F64_BM - 1) / F64_BM, (Cout + F64_BN - 1) / F64_BN, N - n0 < F64_MAX_Z ? N - n0 : F64_MAX_Z);
        f64_gemm_kernel<F64FwdOp><<<grid, F64_THREADS, 0, st>>>(op);
    }
    return check_launch(who);
}

struct F64BwdWs {
    size_t per_image;           // gcol bytes of one image
    size_t gcol, part;          // bytes of the input side (gcol of `chunk` images) and of the grad_weight partials
    int chunk;                  // images per gcol pass at the minimum workspace
    int q_per_split, splits;    // grad_weight split-K over the N*Ho*Wo pixels (shapes only: reproducible everywhere)
    // workspace of a call computing the input side, the parameter side or both (they reuse it one after the other)
    size_t need(bool want_input, bool want_param) const {
        const size_t a = want_input ? gcol : 0, b = want_param ? part : 0;
        return up256(a > b ? a : b);
    }
};
F64BwdWs f64_bwd_ws(int N, int C, int Cout, int K, int HWo) {
    F64BwdWs w;
    w.per_image = static_cast<size_t>(C) * K * HWo * 8;
    size_t chunk = F64_GCOL_BYTES / w.per_image;
    if (chunk > static_cast<size_t>(N)) chunk = N;
    if (chunk > static_cast<size_t>(F64_MAX_Z)) chunk = F64_MAX_Z;
    w.chunk = chunk < 1 ? 1 : static_cast<int>(chunk);
    const long long Q = static_cast<long long>(N) * HWo;
    long long qps = (Q + 31) / 32;
    if (qps < 2048) qps = 2048;
    w.q_per_split = static_cast<int>((qps + F64_BK - 1) / F64_BK * F64_BK);
    w.splits = static_cast<int>((Q + w.q_per_split - 1) / w.q_per_split);
    w.gcol = w.chunk * w.per_image;
    w.part = static_cast<size_t>(w.splits) * Cout * C * K * 8;
    return w;
}

size_t f64_bwd_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, Geo2 g, bool want_input, bool want_param) {
    if (N < 1 || C < 1 || H < 1 || W < 1 || Cout < 1 || kh < 1 || kw < 1 || g.sh < 1 || g.sw < 1 || g.dh < 1 || g.dw < 1)
        return 256;
    const int Ho = (H + 2 * g.ph - (g.dh * (kh - 1) + 1)) / g.sh + 1;
    const int Wo = (W + 2 * g.pw - (g.dw * (kw - 1) + 1)) / g.sw + 1;
    if (Ho < 1 || Wo < 1) return 256;
    return f64_bwd_ws(N, C, Cout, kh * kw, Ho * Wo).need(want_input, want_param);
}

// `want_input` -> grad_x, grad_offset (and grad_mask when mask != NULL), overwritten; `want_param` ->
// grad_weight += scale * dW, grad_bias += db.  The two sides share the workspace one after the other.
int f64_backward_impl(const char* who, const double* x, const double* offset, const double* mask, const double* weight,
                      const double* grad_out, double* grad_x, double* grad_offset, double* grad_mask, double* grad_weight,
                      double* grad_bias, double scale, bool want_input, bool want_param, int N, int C, int H, int W, int Cout,
                      int kh, int kw, Geo2 g, int groups, int dg, void* workspace, size_t workspace_bytes, void* stream) {
    if (N == 0 && C > 0 && H > 0 && W > 0 && Cout > 0) return EB_OK;
    const bool ptrs_ok = x && offset && grad_out && (!want_input || (weight && grad_x && grad_offset)) &&
                         (!want_param || grad_weight);
    F64Geom G;
    if (int rc = f64_check(who, ptrs_ok, N, C, H, W, Cout, kh, kw, g, groups, dg, &G)) return rc;
    const int K = kh * kw, HWo = G.Ho * G.Wo, CK = C * K;
    const F64BwdWs ws = f64_bwd_ws(N, C, Cout, K, HWo);
    const size_t need = ws.need(want_input, want_param);
    if (!workspace || workspace_bytes < need)
        return fail(EB_ERR_WORKSPACE, "%s: workspace %zu < %zu", who, workspace_bytes, need);
    if (!al16(workspace)) return fail(EB_ERR_ALIGNMENT, "%s: workspace must be 16-byte aligned", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* buf = static_cast<double*>(workspace);
    if (want_input) {
        cudaMemsetAsync(grad_x, 0, static_cast<size_t>(N) * C * H * W * 8, st);
        size_t fit = workspace_bytes / ws.per_image;             // a larger workspace takes more images per pass
        int chunk = fit > static_cast<size_t>(N) ? N : static_cast<int>(fit);
        if (chunk > F64_MAX_Z) chunk = F64_MAX_Z;
        if (chunk < ws.chunk) chunk = ws.chunk;
        F64GcolOp op;
        op.G = G; op.weight = weight; op.grad_out = grad_out; op.gcol = buf; op.M = HWo; op.N = CK;
        for (int n0 = 0; n0 < N; n0 += chunk) {
            const int nc = N - n0 < chunk ? N - n0 : chunk;
            op.n_first = n0;
            f64_gemm_kernel<F64GcolOp><<<dim3((HWo + F64_BM - 1) / F64_BM, (CK + F64_BN - 1) / F64_BN, nc), F64_THREADS, 0, st>>>(op);
            f64_coord_scatter_kernel<<<grid_1d(static_cast<long long>(nc) * dg * K * HWo, 256), 256, 0, st>>>(
                G, x, offset, mask, buf, n0, nc, grad_x, grad_offset, mask ? grad_mask : nullptr);
        }
        if (int rc = check_launch(who)) return rc;
    }
    if (want_param) {
        F64WgradOp op;
        op.G = G; op.x = x; op.offset = offset; op.mask = mask; op.grad_out = grad_out; op.part = buf;
        op.M = Cout; op.N = CK; op.q_per_split = ws.q_per_split; op.Q = N * HWo;
        f64_gemm_kernel<F64WgradOp><<<dim3((Cout + F64_BM - 1) / F64_BM, (CK + F64_BN - 1) / F64_BN, ws.splits), F64_THREADS, 0, st>>>(op);
        const long long n = static_cast<long long>(Cout) * CK;
        f64_wgrad_reduce_kernel<<<grid_1d(n, 256), 256, 0, st>>>(buf, ws.splits, n, scale, grad_weight);
        if (grad_bias) f64_bias_kernel<<<Cout, 256, 0, st>>>(grad_out, grad_bias, N, Cout, HWo);
        if (int rc = check_launch(who)) return rc;
    }
    return EB_OK;
}
}  // namespace

int eb_mdcn_forward_f64(const double* x, const double* offset, const double* mask, const double* weight, const double* bias,
                        double* out, int N, int C, int H, int W, int Cout, int kh, int kw, int stride, int pad, int dil,
                        int groups, int dg, void* stream) {
    return f64_forward_impl("mdcn_forward_f64", x, offset, mask, weight, bias, out, N, C, H, W, Cout, kh, kw,
                            Geo2{stride, stride, pad, pad, dil, dil}, groups, dg, stream, true);
}

int eb_dcn1_forward_f64(const double* x, const double* offset, const double* weight, double* out, int N, int C, int H, int W,
                        int Cout, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                        int groups, int dg, void* stream) {
    return f64_forward_impl("dcn1_forward_f64", x, offset, nullptr, weight, nullptr, out, N, C, H, W, Cout, kh, kw,
                            Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, groups, dg, stream, false);
}

size_t eb_mdcn_backward_f64_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride, int pad, int dil) {
    return f64_bwd_workspace(N, C, H, W, Cout, kh, kw, Geo2{stride, stride, pad, pad, dil, dil}, true, true);
}

size_t eb_dcn1_backward_input_f64_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h, int stride_w,
                                            int pad_h, int pad_w, int dil_h, int dil_w) {
    return f64_bwd_workspace(N, C, H, W, Cout, kh, kw, Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, true, false);
}

size_t eb_dcn1_backward_parameters_f64_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h,
                                                 int stride_w, int pad_h, int pad_w, int dil_h, int dil_w) {
    return f64_bwd_workspace(N, C, H, W, Cout, kh, kw, Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, false, true);
}

int eb_mdcn_backward_f64(const double* x, const double* offset, const double* mask, const double* weight,
                         const double* grad_out, double* grad_x, double* grad_offset, double* grad_mask, double* grad_weight,
                         double* grad_bias, int N, int C, int H, int W, int Cout, int kh, int kw, int stride, int pad, int dil,
                         int groups, int dg, void* workspace, size_t workspace_bytes, void* stream) {
    if (!(N == 0) && (!mask || !grad_mask)) return fail(EB_ERR_NULLPTR, "mdcn_backward_f64: null pointer");
    return f64_backward_impl("mdcn_backward_f64", x, offset, mask, weight, grad_out, grad_x, grad_offset, grad_mask,
                             grad_weight, grad_bias, 1.0, true, true, N, C, H, W, Cout, kh, kw,
                             Geo2{stride, stride, pad, pad, dil, dil}, groups, dg, workspace, workspace_bytes, stream);
}

int eb_dcn1_backward_input_f64(const double* x, const double* offset, const double* weight, const double* grad_out,
                               double* grad_x, double* grad_offset, int N, int C, int H, int W, int Cout, int kh, int kw,
                               int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int groups, int dg,
                               void* workspace, size_t workspace_bytes, void* stream) {
    return f64_backward_impl("dcn1_backward_input_f64", x, offset, nullptr, weight, grad_out, grad_x, grad_offset, nullptr,
                             nullptr, nullptr, 1.0, true, false, N, C, H, W, Cout, kh, kw,
                             Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, groups, dg, workspace, workspace_bytes, stream);
}

int eb_dcn1_backward_parameters_f64(const double* x, const double* offset, const double* grad_out, double* grad_weight,
                                    double scale, int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h,
                                    int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int groups, int dg,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    return f64_backward_impl("dcn1_backward_parameters_f64", x, offset, nullptr, nullptr, grad_out, nullptr, nullptr, nullptr,
                             grad_weight, nullptr, scale, false, true, N, C, H, W, Cout, kh, kw,
                             Geo2{stride_h, stride_w, pad_h, pad_w, dil_h, dil_w}, groups, dg, workspace, workspace_bytes, stream);
}

// ---- layout / elementwise ---------------------------------------------------------------------
int eb_nchw_f32_to_nhwc_f16(const float* src, void* dst, int N, int C, int H, int W, int dst_pix_stride,
                            int dst_ch_off, void* stream) {
    if (!src || !dst) return fail(EB_ERR_NULLPTR, "nchw_to_nhwc: null pointer");
    if (N < 0 || C < 1 || H < 1 || W < 1 || dst_pix_stride < C + dst_ch_off) return fail(EB_ERR_INVALID_SHAPE, "nchw_to_nhwc");
    if (N == 0) return EB_OK;
    dim3 grid((H * W + 31) / 32, (C + 31) / 32, N), block(32, 8);
    nchw_f32_to_nhwc_f16_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
        src, static_cast<__half*>(dst), C, H * W, dst_pix_stride, dst_ch_off);
    return check_launch("nchw_to_nhwc");
}

int eb_nhwc_f16_to_nchw_f32(const void* src, int src_pix_stride, int src_ch_off, float* dst, int N, int C,
                            int H, int W, void* stream) {
    if (!src || !dst) return fail(EB_ERR_NULLPTR, "nhwc_to_nchw: null pointer");
    if (N < 0 || C < 1 || H < 1 || W < 1 || src_pix_stride < C + src_ch_off) return fail(EB_ERR_INVALID_SHAPE, "nhwc_to_nchw");
    if (N == 0) return EB_OK;
    dim3 grid((H * W + 31) / 32, (C + 31) / 32, N), block(32, 8);
    nhwc_f16_to_nchw_f32_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(src), dst, C, H * W, src_pix_stride, src_ch_off);
    return check_launch("nhwc_to_nchw");
}

int eb_conv_first(const float* x, const float* w, const float* bias, void* out, int N, int H, int W, int Cout,
                  int out_pix_stride, int act, void* stream) {
    if (!x || !w || !out) return fail(EB_ERR_NULLPTR, "conv_first: null pointer");
    if (N < 0 || H < 1 || W < 1 || Cout < 8 || Cout % 8 || Cout > 512 || out_pix_stride % 8 || out_pix_stride < Cout || !al16(out))
        return fail(EB_ERR_INVALID_SHAPE, "conv_first: shape");
    if (N == 0) return EB_OK;
    const int smem = Cout * 28 * 4;
    if (int rc = set_smem(conv_first_kernel, smem)) return rc;
    const long long items = static_cast<long long>(N) * H * ((W + 3) / 4) * (Cout / 8);
    conv_first_kernel<<<grid_1d(items, 256), 256, smem, static_cast<cudaStream_t>(stream)>>>(
        x, w, bias, static_cast<__half*>(out), N, H, W, Cout, out_pix_stride, act);
    return check_launch("conv_first");
}

int eb_conv_last(const void* x, int x_pix_stride, const float* w, const float* bias, const float* base,
                 long long base_img_stride, int scale, float* out, int N, int H, int W, int Cin, void* stream) {
    if (!x || !w || !base || !out) return fail(EB_ERR_NULLPTR, "conv_last: null pointer");
    if (N < 0 || H < 1 || W < 1 || Cin < 8 || Cin % 8 || Cin > 512 || x_pix_stride % 8 || x_pix_stride < Cin || !al16(x) ||
        (scale != 1 && scale != 4) || H % scale || W % scale)
        return fail(EB_ERR_INVALID_SHAPE, "conv_last: shape");
    if (N == 0) return EB_OK;
    const int smem = 27 * Cin * 4;
    if (int rc = set_smem(conv_last_kernel, smem)) return rc;
    const long long items = static_cast<long long>(N) * H * ((W + 3) / 4);
    conv_last_kernel<<<grid_1d(items, 128), 128, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x), x_pix_stride, w, bias, base, base_img_stride, scale, out, N, H, W, Cin);
    return check_launch("conv_last");
}

int eb_add_base(const float* base, long long base_img_stride, int scale, float* out, int N, int C, int H, int W, void* stream) {
    if (!base || !out) return fail(EB_ERR_NULLPTR, "add_base: null pointer");
    if (N < 0 || C < 1 || H < 1 || W < 1 || (scale != 1 && scale != 4) || H % scale || W % scale)
        return fail(EB_ERR_INVALID_SHAPE, "add_base: shape");
    if (N == 0) return EB_OK;
    add_base_kernel<<<grid_1d(static_cast<long long>(N) * C * H * W, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        base, base_img_stride, scale, out, N, C, H, W);
    return check_launch("add_base");
}

static bool view_ok(const void* p, int ps, int co, int C) {
    return p && al16(p) && ps % 8 == 0 && co % 8 == 0 && C % 8 == 0 && ps >= co + C;
}

int eb_upsample2x(const void* src, int sps, int sco, void* dst, int dps, int dco, int N, int H, int W, int C,
                  float mul, const void* add, int aps, int aco, void* stream) {
    if (!view_ok(src, sps, sco, C) || !view_ok(dst, dps, dco, C) || (add && !view_ok(add, aps, aco, C)))
        return fail(EB_ERR_ALIGNMENT, "upsample2x: bad view");
    if (N < 0 || H < 1 || W < 1) return fail(EB_ERR_INVALID_SHAPE, "upsample2x: shape");
    if (N == 0) return EB_OK;
    const long long per_img = static_cast<long long>(H) * W * (C / 8);
    if (per_img > 0x7fffffffll || N > 65535) return fail(EB_ERR_INVALID_SHAPE, "upsample2x: image too large for 32-bit indexing");
    const long long blocks = (per_img + 255) / 256;
    const dim3 grid(static_cast<unsigned>(blocks < 65535 * 4 ? blocks : 65535 * 4), static_cast<unsigned>(N));
    upsample2x_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(src), sps, sco, static_cast<__half*>(dst), dps, dco, H, W, C, mul,
        static_cast<const __half*>(add), aps, aco);
    return check_launch("upsample2x");
}

// ---- frame staging either side of the network (read_img_seq / tensor2img arithmetic, bit-exact; elementwise.cuh)
int eb_frames_u8_to_f32(const void* hwc_u8, float* chw_f32, int N, int H, int W, int bgr2rgb, void* stream) {
    if (!hwc_u8 || !chw_f32) return fail(EB_ERR_NULLPTR, "frames_u8_to_f32: null pointer");
    if (N < 0 || H < 1 || W < 1 || static_cast<long long>(H) * W > 0x7fffffffll) return fail(EB_ERR_INVALID_SHAPE, "frames_u8_to_f32: N=%d H=%d W=%d", N, H, W);
    if (N == 0) return EB_OK;
    const long long total = static_cast<long long>(N) * H * W;
    frames_u8_to_f32_kernel<<<grid_1d(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint8_t*>(hwc_u8), chw_f32, H * W, total, bgr2rgb ? 1 : 0);
    return check_launch("frames_u8_to_f32");
}

int eb_tensor2img_u8(const float* chw_f32, void* hwc_u8, int N, int C, int H, int W, int rgb2bgr, float lo, float hi, void* stream) {
    if (!chw_f32 || !hwc_u8) return fail(EB_ERR_NULLPTR, "tensor2img_u8: null pointer");
    if (N < 0 || (C != 1 && C != 3) || H < 1 || W < 1 || static_cast<long long>(H) * W > 0x7fffffffll || !(hi > lo))
        return fail(EB_ERR_INVALID_SHAPE, "tensor2img_u8: N=%d C=%d H=%d W=%d range [%g, %g]", N, C, H, W, lo, hi);
    if (N == 0) return EB_OK;
    const long long total = static_cast<long long>(N) * H * W;
    tensor2img_u8_kernel<<<grid_1d(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        chw_f32, static_cast<uint8_t*>(hwc_u8), C, H * W, total, rgb2bgr ? 1 : 0, lo, hi);
    return check_launch("tensor2img_u8");
}

int eb_pool_max_avg(const void* src, int sps, int sco, void* dst, int dps, int dco, int N, int H, int W, int C,
                    void* stream) {
    if (!view_ok(src, sps, sco, C) || !view_ok(dst, dps, dco, 2 * C)) return fail(EB_ERR_ALIGNMENT, "pool: bad view");
    if (N < 0 || H < 1 || W < 1) return fail(EB_ERR_INVALID_SHAPE, "pool: shape");
    if (N == 0) return EB_OK;
    const long long items = static_cast<long long>(N) * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8);
    pool_max_avg_kernel<<<grid_1d(items, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(src), sps, sco, static_cast<__half*>(dst), dps, dco, N, H, W, C);
    return check_launch("pool_max_avg");
}

int eb_tsa_temporal(const void* emb, const void* emb_ref, const void* aligned, void* dst, int B, int T, int H,
                    int W, int C, void* stream) {
    if (!emb || !emb_ref || !aligned || !dst) return fail(EB_ERR_NULLPTR, "tsa_temporal: null pointer");
    const int lpp = C / 8;
    if (B < 0 || T < 1 || H < 1 || W < 1 || C % 8 || lpp < 1 || lpp > 32 || (lpp & (lpp - 1)))
        return fail(EB_ERR_INVALID_SHAPE, "tsa_temporal: C=%d must be 8*2^k <= 256", C);
    if (!al16(emb) || !al16(emb_ref) || !al16(aligned) || !al16(dst)) return fail(EB_ERR_ALIGNMENT, "tsa_temporal");
    if (B == 0) return EB_OK;
    const long long items = static_cast<long long>(B) * H * W * lpp;
    tsa_temporal_kernel<<<grid_1d(items, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(emb), static_cast<const __half*>(emb_ref), static_cast<const __half*>(aligned),
        static_cast<__half*>(dst), B, T, H * W, C);
    return check_launch("tsa_temporal");
}

size_t eb_f32_blocked_elems(int N, int H, int W, int C) {
    return static_cast<size_t>(N) * ((H + 15) / 16) * ((W + 15) / 16) * 256 * static_cast<size_t>(C);
}

int eb_tsa_modulate(const void* feat, int fps, int fco, const void* attn, const void* attn_add, void* out16,
                    float* out32, int N, int H, int W, int C, int f32_blocked, void* stream) {
    const long long npix = static_cast<long long>(N) * H * W;
    if (f32_blocked && C % 32) return fail(EB_ERR_UNSUPPORTED, "tsa_modulate: blocked fp32 output needs C %% 32 == 0");
    if (!view_ok(feat, fps, fco, C) || !attn || !attn_add || (!out16 && !out32) || !al16(attn) || !al16(attn_add) ||
        (out16 && !al16(out16)) || (out32 && !al16(out32)))
        return fail(EB_ERR_ALIGNMENT, "tsa_modulate: bad view");
    if (npix < 0) return fail(EB_ERR_INVALID_SHAPE, "tsa_modulate: npix");
    if (npix == 0) return EB_OK;
    const long long items = npix * (C / 8);
    tsa_modulate_kernel<<<grid_1d(items, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(feat), fps, fco, static_cast<const __half*>(attn),
        static_cast<const __half*>(attn_add), static_cast<__half*>(out16), out32, npix, C, H, W, f32_blocked);
    return check_launch("tsa_modulate");
}

int eb_add(const void* a, int aps, int aco, const void* b, int bps, int bco, void* dst, int dps, int dco, int npix,
           int C, void* stream) {
    if (!view_ok(a, aps, aco, C) || !view_ok(b, bps, bco, C) || !view_ok(dst, dps, dco, C))
        return fail(EB_ERR_ALIGNMENT, "add: bad view");
    if (npix < 0) return fail(EB_ERR_INVALID_SHAPE, "add: npix");
    if (npix == 0) return EB_OK;
    const long long items = static_cast<long long>(npix) * (C / 8);
    add_kernel<<<grid_1d(items, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(a), aps, aco, static_cast<const __half*>(b), bps, bco, static_cast<__half*>(dst),
        dps, dco, npix, C);
    return check_launch("add");
}

}  // extern "C"

// parallel-cnn_b200/csrc/conv_bwd.cu -- weight- and input-gradient of the generic NHWC bf16 convolution (SURVEY.md x3).
//
// Entry points + the general-shape kernels on the fp32 FMA pipe (bf16 operands, fp32 accumulation, deterministic two-stage
// reduction, no atomics).  Shapes the tensor cores can take (64 filters; conv_wgrad_tc.cu, conv_dgrad_tc.cu) are routed to the tcgen05
// kernels, which are the roofline path: both passes move the same 6.6 MB/image as the forward pass (config 5) and are
// HBM-bound at 170 MFLOP per 6.6 MB, which the FMA pipe cannot sustain (SURVEY.md 8d).  PCNN_CONV_BWD=fma forces the
// FMA-pipe kernels (used by the tests to check both paths against the oracle).
//   wgrad  dw[k][r][s][c] = sum_{n,p,q} dy[n][p][q][k] * x[n][p+r][q+s][c]          [ref: layer.h:371-395 without the /576]
//   dgrad  dx[n][h][w][c] = sum_{k,r,s} dy[n][h-r][w-s][k] * f[k][r][s][c]          (the reference never needs it: c1 is the first layer)
// The _strided entry points take a window step st in 1..4 (the forward plan's pcnn_conv_tc_plan_create_strided): x[n][p*st+r][q*st+s][c]
// in the weight gradient, dy[n][(h-r)/st][(w-s)/st][k] over (h-r) % st == 0, (w-s) % st == 0 in the input gradient; the
// stride-1 entry points are that case.
#include "pcnn_internal.h"

#include <cuda_bf16.h>
#include <stdlib.h>

// conv_dgrad_tc.cu
bool pcnn_conv_dgrad_rows_ok(int N, int H, int W, int C, int K, int R, int S, int stride, const void *dy);
int pcnn_conv_dgrad_rows(pcnn_ctx *ctx, const void *dy_bf16, const float *filt_f32_dev, void *dx_bf16, int N, int H, int W, int C, int K,
                         int R, int S, int stride, int row_pitch, int image_rows, int dy_channels = 0);
// conv_wgrad_tc.cu
bool pcnn_conv_wgrad_rows_ok(int N, int H, int W, int C, int K, int R, int S, int stride, int row_pitch, const void *x, const void *dy);
int pcnn_conv_wgrad_rows(pcnn_ctx *ctx, const void *x_bf16, const void *dy_bf16, float *dw_f32, int N, int H, int W, int C, int K,
                         int R, int S, int stride, int row_pitch, int image_rows, int dy_channels = 0);
void pcnn_conv_dgrad_rows_info(int H, int W, int C, int K, int R, int S, int stride, int *out4);
void pcnn_conv_wgrad_rows_info(int H, int W, int C, int K, int R, int S, int stride, int *out4);

namespace {

constexpr int WG_THREADS = 256;
constexpr int WG_MAXO = 20;           // outputs per thread: K*R*S*C <= 5120

struct ConvShape {
    int N, H, W, C, K, R, S, P, Q;
    int row_pitch;                    // elements between rows of x
    int image_rows;                   // rows between images of x
    int stride;                       // window step in both directions
};

__device__ __forceinline__ float bf(const __nv_bfloat16 *p) { return __bfloat162float(*p); }

// one CTA walks output rows (n, p) = blockIdx.x, + gridDim.x, ...; thread t owns outputs t, t + 256, ...
__global__ void __launch_bounds__(WG_THREADS) k_conv_wgrad_partial(const __nv_bfloat16 *__restrict__ x,
                                                                    const __nv_bfloat16 *__restrict__ dy, float *__restrict__ slots,
                                                                    const ConvShape s) {
    const int nout = s.K * s.R * s.S * s.C;
    int k[WG_MAXO], xoff[WG_MAXO];
    float acc[WG_MAXO];
#pragma unroll
    for (int i = 0; i < WG_MAXO; ++i) {
        const int o = threadIdx.x + i * WG_THREADS;
        acc[i] = 0.0f;
        k[i] = 0;
        xoff[i] = -1;
        if (o < nout) {
            const int c = o % s.C, ss = (o / s.C) % s.S, r = (o / (s.C * s.S)) % s.R;
            k[i] = o / (s.C * s.S * s.R);
            xoff[i] = r * s.row_pitch + ss * s.C + c;
        }
    }
    const long rows = (long)s.N * s.P;
    for (long row = blockIdx.x; row < rows; row += gridDim.x) {
        const int n = (int)(row / s.P), p = (int)(row % s.P);
        const __nv_bfloat16 *xr = x + ((long)n * s.image_rows + p * s.stride) * s.row_pitch;
        const __nv_bfloat16 *dr = dy + row * s.Q * s.K;
        const int xstep = s.stride * s.C;
        for (int q = 0; q < s.Q; ++q) {
#pragma unroll
            for (int i = 0; i < WG_MAXO; ++i)
                if (xoff[i] >= 0) acc[i] = fmaf(bf(dr + q * s.K + k[i]), bf(xr + q * xstep + xoff[i]), acc[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < WG_MAXO; ++i) {
        const int o = threadIdx.x + i * WG_THREADS;
        if (o < nout) slots[(long)blockIdx.x * nout + o] = acc[i];
    }
}

__global__ void k_conv_wgrad_reduce(const float *__restrict__ slots, float *__restrict__ dw, int nslots, int nout) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= nout) return;
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
    int k = 0;
    for (; k + 3 < nslots; k += 4) {
        s0 += slots[(long)k * nout + o];
        s1 += slots[(long)(k + 1) * nout + o];
        s2 += slots[(long)(k + 2) * nout + o];
        s3 += slots[(long)(k + 3) * nout + o];
    }
    for (; k < nslots; ++k) s0 += slots[(long)k * nout + o];
    dw[o] = (s0 + s1) + (s2 + s3);
}

// one thread per input element (n, h, w, c)
__global__ void __launch_bounds__(256) k_conv_dgrad(const __nv_bfloat16 *__restrict__ dy, const float *__restrict__ f,
                                                   __nv_bfloat16 *__restrict__ dx, const ConvShape s) {
    const long total = (long)s.N * s.H * s.W * s.C;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % s.C);
        const int w = (int)((idx / s.C) % s.W);
        const int h = (int)((idx / ((long)s.C * s.W)) % s.H);
        const int n = (int)(idx / ((long)s.C * s.W * s.H));
        float acc = 0.0f;
        for (int r = 0; r < s.R; ++r) {
            if (h - r < 0 || (h - r) % s.stride) continue;
            const int p = (h - r) / s.stride;
            if (p >= s.P) continue;
            for (int ss = 0; ss < s.S; ++ss) {
                if (w - ss < 0 || (w - ss) % s.stride) continue;
                const int q = (w - ss) / s.stride;
                if (q >= s.Q) continue;
                const __nv_bfloat16 *d = dy + (((long)n * s.P + p) * s.Q + q) * s.K;
                const float *fp = f + ((long)r * s.S + ss) * s.C + c;
                for (int k = 0; k < s.K; ++k) acc = fmaf(bf(d + k), fp[(long)k * s.R * s.S * s.C], acc);
            }
        }
        dx[((long)n * s.image_rows + h) * s.row_pitch + w * s.C + c] = __float2bfloat16_rn(acc);
    }
}

// dy [rows][K] -> [rows][Kp] bf16 with zero filter channels K..Kp-1 (the padded tensor-core path below)
__global__ void __launch_bounds__(256) k_pad_channels_bf16(const __nv_bfloat16 *__restrict__ src, __nv_bfloat16 *__restrict__ dst, long rows,
                                                           int K, int Kp) {
    const long total = rows * (Kp / 8);                       // 16-byte pieces of the destination
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long r = i / (Kp / 8);
        const int k0 = (int)(i % (Kp / 8)) * 8;
        __align__(16) __nv_bfloat16 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = k0 + u < K ? src[r * K + k0 + u] : __float2bfloat16_rn(0.0f);
        *reinterpret_cast<uint4 *>(dst + r * Kp + k0) = *reinterpret_cast<const uint4 *>(v);
    }
}
// filters [K][RSC] fp32 -> [Kp][RSC] with zero filters K..Kp-1
__global__ void k_pad_filters_f32(const float *__restrict__ src, float *__restrict__ dst, int K, int Kp, int rsc) {
    const int total = Kp * rsc;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) dst[i] = i < K * rsc ? src[i] : 0.0f;
}

// second grow-only device scratch (the tensor-core kernels use the first one themselves while they read this one)
int scratch2(pcnn_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->scratch2_bytes) {
        PCNN_CUDA(cudaStreamSynchronize(ctx->stream));
        if (ctx->scratch2) PCNN_CUDA(cudaFree(ctx->scratch2));
        ctx->scratch2 = nullptr;
        ctx->scratch2_bytes = 0;
        const size_t want = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
        PCNN_CUDA(cudaMalloc(&ctx->scratch2, want));
        ctx->scratch2_bytes = want;
    }
    *out = ctx->scratch2;
    return PCNN_OK;
}

// Filter counts that are not a multiple of 64 (LeNet's own 6, a C3-style 16, ...): pad the filter dimension of dy with zero
// channels up to the next multiple of 64 and run the 64-filter tensor-core kernels -- one extra pass that writes Kp / K times the
// bytes of dy, after which the kernel streams the padded tensor: roughly K / (2 Kp) of the roofline of the dense case (K = 32:
// a quarter, K = 6: a twentieth), still 5-25 x the FMA-pipe reference kernels.
int pad_dy(pcnn_ctx *ctx, const void *dy_bf16, long rows, int K, int Kp, size_t extra_bytes, __nv_bfloat16 **dyp, void **extra) {
    const size_t dy_bytes = ((size_t)rows * Kp * 2 + 255) & ~(size_t)255;
    void *base = nullptr;
    int rc = scratch2(ctx, dy_bytes + extra_bytes, &base);
    if (rc) return rc;
    *dyp = reinterpret_cast<__nv_bfloat16 *>(base);
    if (extra) *extra = reinterpret_cast<char *>(base) + dy_bytes;
    const long pieces = rows * (Kp / 8);
    long blocks = (pieces + 255) / 256;
    if (blocks > (long)ctx->sm_count * 16) blocks = (long)ctx->sm_count * 16;
    k_pad_channels_bf16<<<(int)blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const __nv_bfloat16 *>(dy_bf16), *dyp, rows, K, Kp);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}

int check_shape(const char *fn, int N, int H, int W, int C, int K, int R, int S, int stride, int row_pitch, int image_rows, ConvShape *out) {
    PCNN_REQUIRE(N > 0 && C > 0 && K > 0 && R > 0 && S > 0 && H >= R && W >= S, PCNN_ERR_ARG, "%s: bad shape", fn);
    PCNN_REQUIRE(stride >= 1 && stride <= 4, PCNN_ERR_ARG, "%s: stride %d outside 1..4", fn, stride);
    if (row_pitch <= 0) row_pitch = W * C;
    if (image_rows <= 0) image_rows = H;
    PCNN_REQUIRE(row_pitch >= W * C && image_rows >= H, PCNN_ERR_ARG, "%s: pitches smaller than the image", fn);
    out->N = N; out->H = H; out->W = W; out->C = C; out->K = K; out->R = R; out->S = S;
    out->P = (H - R) / stride + 1; out->Q = (W - S) / stride + 1; out->row_pitch = row_pitch; out->image_rows = image_rows;
    out->stride = stride;
    return PCNN_OK;
}

int conv_wgrad(const char *fn, pcnn_ctx *ctx, const void *x_bf16, const void *dy_bf16, float *dw_f32, int N, int H, int W, int C, int K, int R,
               int S, int stride, int row_pitch, int image_rows) {
    PCNN_REQUIRE(ctx && x_bf16 && dy_bf16 && dw_f32, PCNN_ERR_ARG, "%s: NULL argument", fn);
    ConvShape s;
    int rc = check_shape(fn, N, H, W, C, K, R, S, stride, row_pitch, image_rows, &s);
    if (rc) return rc;
    if (ctx->conv_bwd_path == PCNN_CONV_BWD_TENSOR) {
        const int Kp = (K + 63) / 64 * 64;
        if (K % 64 && Kp <= 256 && pcnn_conv_wgrad_rows_ok(N, H, W, C, Kp, R, S, stride, s.row_pitch, x_bf16, nullptr)) {
            pcnn_device_guard g(ctx->device);
            __nv_bfloat16 *dyp = nullptr;
            void *dwp = nullptr;
            const int rsc = R * S * C;
            // K a multiple of 8 (16-byte pixel pitch) and 16-byte aligned: dy is read in place, the TMA zero-fills filters
            // K..63 of every box; otherwise (LeNet's 6 filters) one pass builds a zero-padded copy first
            const bool in_place = K % 8 == 0 && ((uintptr_t)dy_bf16 & 15) == 0;
            if (in_place) {
                void *base = nullptr;
                if ((rc = scratch2(ctx, (size_t)Kp * rsc * sizeof(float), &base))) return rc;
                dwp = base;
            } else if ((rc = pad_dy(ctx, dy_bf16, (long)N * s.P * s.Q, K, Kp, (size_t)Kp * rsc * sizeof(float), &dyp, &dwp))) {
                return rc;
            }
            if ((rc = pcnn_conv_wgrad_rows(ctx, x_bf16, in_place ? dy_bf16 : dyp, reinterpret_cast<float *>(dwp), N, H, W, C, Kp, R, S,
                                           stride, s.row_pitch, s.image_rows, in_place ? K : 0)))
                return rc;
            PCNN_CUDA(cudaMemcpyAsync(dw_f32, dwp, (size_t)K * rsc * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));   // filters 0..K-1
            return PCNN_OK;
        }
        PCNN_REQUIRE(pcnn_conv_wgrad_rows_ok(N, H, W, C, K, R, S, stride, s.row_pitch, x_bf16, dy_bf16), PCNN_ERR_ARG,
                     "%s: no tensor-core kernel for C = %d, K = %d, %dx%d taps, stride %d (needs K <= 256 -- padded to a multiple of 64 --, "
                     "((RB - 1) * stride + R) * S * C <= 64, a row pitch that is a multiple of 8 elements, 16-byte aligned operands); the FMA-pipe "
                     "reference kernels (~1 %% of the HBM roofline) must be selected explicitly with pcnn_conv_bwd_select(ctx, PCNN_CONV_BWD_REFERENCE)",
                     fn, C, K, R, S, stride);
        return pcnn_conv_wgrad_rows(ctx, x_bf16, dy_bf16, dw_f32, N, H, W, C, K, R, S, stride, s.row_pitch, s.image_rows);
    }
    const int nout = K * R * S * C;
    PCNN_REQUIRE(nout <= WG_THREADS * WG_MAXO, PCNN_ERR_ARG, "%s: K*R*S*C = %d exceeds %d", fn, nout, WG_THREADS * WG_MAXO);
    pcnn_device_guard g(ctx->device);
    const long rows = (long)N * s.P;
    int grid = (int)(rows < (long)ctx->sm_count * 8 ? rows : (long)ctx->sm_count * 8);
    float *slots = nullptr;
    if ((rc = pcnn_scratch(ctx, (size_t)grid * nout * sizeof(float), (void **)&slots))) return rc;
    k_conv_wgrad_partial<<<grid, WG_THREADS, 0, ctx->stream>>>(reinterpret_cast<const __nv_bfloat16 *>(x_bf16),
                                                              reinterpret_cast<const __nv_bfloat16 *>(dy_bf16), slots, s);
    PCNN_CHECK_LAUNCH(ctx);
    k_conv_wgrad_reduce<<<(nout + 127) / 128, 128, 0, ctx->stream>>>(slots, dw_f32, grid, nout);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}

int conv_dgrad(const char *fn, pcnn_ctx *ctx, const void *dy_bf16, const float *filt_f32_dev, void *dx_bf16, int N, int H, int W, int C, int K,
               int R, int S, int stride, int row_pitch, int image_rows) {
    PCNN_REQUIRE(ctx && dy_bf16 && filt_f32_dev && dx_bf16, PCNN_ERR_ARG, "%s: NULL argument", fn);
    ConvShape s;
    int rc = check_shape(fn, N, H, W, C, K, R, S, stride, row_pitch, image_rows, &s);
    if (rc) return rc;
    if (ctx->conv_bwd_path == PCNN_CONV_BWD_TENSOR) {
        const int Kp = (K + 63) / 64 * 64;
        if (K % 64 && Kp <= 256 && pcnn_conv_dgrad_rows_ok(N, H, W, C, Kp, R, S, stride, nullptr)) {
            pcnn_device_guard g(ctx->device);
            __nv_bfloat16 *dyp = nullptr;
            void *fp = nullptr;
            const int rsc = R * S * C;
            const bool in_place = K % 8 == 0 && ((uintptr_t)dy_bf16 & 15) == 0;      // see pcnn_conv_wgrad
            if (in_place) {
                void *base = nullptr;
                if ((rc = scratch2(ctx, (size_t)Kp * rsc * sizeof(float), &base))) return rc;
                fp = base;
            } else if ((rc = pad_dy(ctx, dy_bf16, (long)N * s.P * s.Q, K, Kp, (size_t)Kp * rsc * sizeof(float), &dyp, &fp))) {
                return rc;
            }
            k_pad_filters_f32<<<(Kp * rsc + 255) / 256, 256, 0, ctx->stream>>>(filt_f32_dev, reinterpret_cast<float *>(fp), K, Kp, rsc);
            PCNN_CHECK_LAUNCH(ctx);
            return pcnn_conv_dgrad_rows(ctx, in_place ? dy_bf16 : dyp, reinterpret_cast<const float *>(fp), dx_bf16, N, H, W, C, Kp, R, S,
                                        stride, s.row_pitch, s.image_rows, in_place ? K : 0);
        }
        PCNN_REQUIRE(pcnn_conv_dgrad_rows_ok(N, H, W, C, K, R, S, stride, dy_bf16), PCNN_ERR_ARG,
                     "%s: no tensor-core kernel for C = %d, K = %d, %dx%d taps, stride %d (needs K <= 256 -- padded to a multiple of 64 -- and, "
                     "at strides 1 and 2, 3x3 taps with C in {1,2,3,4,8}, 5x5 with C in {1,3} or 7x7 with C = 1; at stride 3, 3x3 with C in "
                     "{1,2,3}; at stride 4, 3x3 with C = 3 or 5x5 with C = 1); the FMA-pipe reference kernels (~1 %% of the HBM roofline) must "
                     "be selected explicitly with pcnn_conv_bwd_select(ctx, PCNN_CONV_BWD_REFERENCE)", fn, C, K, R, S, stride);
        return pcnn_conv_dgrad_rows(ctx, dy_bf16, filt_f32_dev, dx_bf16, N, H, W, C, K, R, S, stride, s.row_pitch, s.image_rows);
    }
    pcnn_device_guard g(ctx->device);
    const long total = (long)N * H * W * C;
    long blocks = (total + 255) / 256;
    if (blocks > (long)ctx->sm_count * 16) blocks = (long)ctx->sm_count * 16;
    k_conv_dgrad<<<(int)blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const __nv_bfloat16 *>(dy_bf16), filt_f32_dev,
                                                      reinterpret_cast<__nv_bfloat16 *>(dx_bf16), s);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}

}  // namespace

extern "C" int pcnn_conv_wgrad(pcnn_ctx *ctx, const void *x_bf16, const void *dy_bf16, float *dw_f32, int N, int H, int W, int C,
                               int K, int R, int S, int row_pitch, int image_rows) {
    return conv_wgrad("pcnn_conv_wgrad", ctx, x_bf16, dy_bf16, dw_f32, N, H, W, C, K, R, S, 1, row_pitch, image_rows);
}

extern "C" int pcnn_conv_wgrad_strided(pcnn_ctx *ctx, const void *x_bf16, const void *dy_bf16, float *dw_f32, int N, int H, int W, int C,
                                       int K, int R, int S, int stride, int row_pitch, int image_rows) {
    return conv_wgrad("pcnn_conv_wgrad_strided", ctx, x_bf16, dy_bf16, dw_f32, N, H, W, C, K, R, S, stride, row_pitch, image_rows);
}

extern "C" int pcnn_conv_dgrad(pcnn_ctx *ctx, const void *dy_bf16, const float *filt_f32_dev, void *dx_bf16, int N, int H, int W,
                               int C, int K, int R, int S, int row_pitch, int image_rows) {
    return conv_dgrad("pcnn_conv_dgrad", ctx, dy_bf16, filt_f32_dev, dx_bf16, N, H, W, C, K, R, S, 1, row_pitch, image_rows);
}

extern "C" int pcnn_conv_dgrad_strided(pcnn_ctx *ctx, const void *dy_bf16, const float *filt_f32_dev, void *dx_bf16, int N, int H, int W,
                                       int C, int K, int R, int S, int stride, int row_pitch, int image_rows) {
    return conv_dgrad("pcnn_conv_dgrad_strided", ctx, dy_bf16, filt_f32_dev, dx_bf16, N, H, W, C, K, R, S, stride, row_pitch, image_rows);
}

extern "C" int pcnn_conv_bwd_select(pcnn_ctx *ctx, int path) {
    PCNN_REQUIRE(ctx, PCNN_ERR_ARG, "pcnn_conv_bwd_select: ctx is NULL");
    PCNN_REQUIRE(path == PCNN_CONV_BWD_TENSOR || path == PCNN_CONV_BWD_REFERENCE, PCNN_ERR_ARG, "pcnn_conv_bwd_select: bad path %d", path);
    ctx->conv_bwd_path = path;
    return PCNN_OK;
}

// ---- zero padding around NHWC bf16 images (SURVEY.md 8f row 4: the "same"-padding front-end of the valid-padding kernels) ----
namespace {

// dst[n][h + ph][(w + pw) * C + c] = src[n][h][w][c]; everything else of the [dst_image_rows x dst_pitch] canvas = 0.
// One thread per 2 destination elements (4-byte stores); rows are walked by a grid-stride loop.
__global__ void __launch_bounds__(256) k_pad_nhwc(const __nv_bfloat16 *__restrict__ src, __nv_bfloat16 *__restrict__ dst, int N, int H,
                                                  int W, int C, int ph, int pw, int dst_pitch, int dst_image_rows) {
    const long total = (long)N * dst_image_rows * dst_pitch;
    const int wc = W * C, off = pw * C;
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int col = (int)(i % dst_pitch);
        const long row = i / dst_pitch;
        const int r = (int)(row % dst_image_rows), n = (int)(row / dst_image_rows);
        const int h = r - ph, e = col - off;
        __nv_bfloat16 v = __float2bfloat16_rn(0.0f);
        if (h >= 0 && h < H && e >= 0 && e < wc) v = src[((long)n * H + h) * wc + e];
        dst[i] = v;
    }
}
// the inverse: dst[n][h][w][c] = src[n][h + ph][(w + pw) * C + c]
__global__ void __launch_bounds__(256) k_crop_nhwc(const __nv_bfloat16 *__restrict__ src, __nv_bfloat16 *__restrict__ dst, int N, int H,
                                                   int W, int C, int ph, int pw, int src_pitch, int src_image_rows) {
    const int wc = W * C;
    const long total = (long)N * H * wc;
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int e = (int)(i % wc);
        const long row = i / wc;
        const int h = (int)(row % H), n = (int)(row / H);
        dst[i] = src[((long)n * src_image_rows + h + ph) * src_pitch + pw * C + e];
    }
}

}  // namespace

extern "C" int pcnn_pad_nhwc_bf16(pcnn_ctx *ctx, const void *src_bf16, void *dst_bf16, int N, int H, int W, int C, int pad_h, int pad_w,
                                  int dst_row_pitch, int dst_image_rows) {
    PCNN_REQUIRE(ctx && src_bf16 && dst_bf16 && N > 0 && H > 0 && W > 0 && C > 0 && pad_h >= 0 && pad_w >= 0, PCNN_ERR_ARG,
                 "pcnn_pad_nhwc_bf16: bad argument");
    if (dst_row_pitch <= 0) dst_row_pitch = (W + 2 * pad_w) * C;
    if (dst_image_rows <= 0) dst_image_rows = H + 2 * pad_h;
    PCNN_REQUIRE(dst_row_pitch >= (W + 2 * pad_w) * C && dst_image_rows >= H + 2 * pad_h, PCNN_ERR_ARG,
                 "pcnn_pad_nhwc_bf16: destination canvas smaller than the padded image");
    pcnn_device_guard g(ctx->device);
    const long total = (long)N * dst_image_rows * dst_row_pitch;
    long blocks = (total + 255) / 256;
    if (blocks > (long)ctx->sm_count * 16) blocks = (long)ctx->sm_count * 16;
    k_pad_nhwc<<<(int)blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const __nv_bfloat16 *>(src_bf16), reinterpret_cast<__nv_bfloat16 *>(dst_bf16),
                                                    N, H, W, C, pad_h, pad_w, dst_row_pitch, dst_image_rows);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}

extern "C" int pcnn_crop_nhwc_bf16(pcnn_ctx *ctx, const void *src_bf16, void *dst_bf16, int N, int H, int W, int C, int pad_h, int pad_w,
                                   int src_row_pitch, int src_image_rows) {
    PCNN_REQUIRE(ctx && src_bf16 && dst_bf16 && N > 0 && H > 0 && W > 0 && C > 0 && pad_h >= 0 && pad_w >= 0, PCNN_ERR_ARG,
                 "pcnn_crop_nhwc_bf16: bad argument");
    if (src_row_pitch <= 0) src_row_pitch = (W + 2 * pad_w) * C;
    if (src_image_rows <= 0) src_image_rows = H + 2 * pad_h;
    PCNN_REQUIRE(src_row_pitch >= (W + 2 * pad_w) * C && src_image_rows >= H + 2 * pad_h, PCNN_ERR_ARG,
                 "pcnn_crop_nhwc_bf16: source canvas smaller than the padded image");
    pcnn_device_guard g(ctx->device);
    const long total = (long)N * H * W * C;
    long blocks = (total + 255) / 256;
    if (blocks > (long)ctx->sm_count * 16) blocks = (long)ctx->sm_count * 16;
    k_crop_nhwc<<<(int)blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const __nv_bfloat16 *>(src_bf16), reinterpret_cast<__nv_bfloat16 *>(dst_bf16),
                                                     N, H, W, C, pad_h, pad_w, src_row_pitch, src_image_rows);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}

// Which kernels the backward entry points would pick for a shape and how they tile it (pure host logic, no device needed):
// out[0] = weight gradient on the tensor cores (0/1), out[1..3] = its dy rows per tile, pixels per tile, stages;
// out[4] = input gradient on the tensor cores (0/1), out[5..8] = its column strips, output pixels per lane quarter,
// TMEM slot groups in flight, stages.  Pointer alignment and row pitch are assumed to qualify (16 bytes, multiple of 8).
// The _strided query takes the window step (1..4); its out9[6] counts dx columns per lane quarter (stride x dy pixels).
extern "C" int pcnn_conv_bwd_plan_info_strided(int N, int H, int W, int C, int K, int R, int S, int stride, int *out9) {
    PCNN_REQUIRE(out9 && N > 0 && H >= R && W >= S && C > 0 && K > 0 && R > 0 && S > 0, PCNN_ERR_ARG, "pcnn_conv_bwd_plan_info: bad argument");
    PCNN_REQUIRE(stride >= 1 && stride <= 4, PCNN_ERR_ARG, "pcnn_conv_bwd_plan_info_strided: stride %d outside 1..4", stride);
    for (int i = 0; i < 9; ++i) out9[i] = 0;
    const void *aligned = reinterpret_cast<const void *>((uintptr_t)256);
    const int Kp = (K + 63) / 64 * 64;          // filter counts are zero-padded to a multiple of 64 (pcnn_conv_wgrad / dgrad)
    if (pcnn_conv_wgrad_rows_ok(N, H, W, C, Kp, R, S, stride, 8, aligned, aligned)) pcnn_conv_wgrad_rows_info(H, W, C, Kp, R, S, stride, out9);
    if (pcnn_conv_dgrad_rows_ok(N, H, W, C, Kp, R, S, stride, aligned)) {
        out9[4] = 1;
        pcnn_conv_dgrad_rows_info(H, W, C, Kp, R, S, stride, out9 + 5);
    }
    return PCNN_OK;
}

extern "C" int pcnn_conv_bwd_plan_info(int N, int H, int W, int C, int K, int R, int S, int *out9) {
    return pcnn_conv_bwd_plan_info_strided(N, H, W, C, K, R, S, 1, out9);
}

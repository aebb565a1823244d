// parallel-cnn_b200/csrc/conv_dgrad_tc.cu -- input gradient of the NHWC bf16 convolution (64 filters), row-streaming formulation.
//
//     dx[n][h][w][c] = sum_{k,r,s} dy[n][h-r][w-s][k] * f[k][r][s][c]
//     (window step st: the sum runs over (h-r) % st == 0, (w-s) % st == 0 with dy[n][(h-r)/st][(w-s)/st][k])
//
// Access pattern first: a first version put 128 dy ROWS of one pixel column on the TMEM lanes (col2im folded into the TMEM
// column offset); its TMA boxes gathered 128-byte pieces of 128 different rows, and a TMA pipeline with that pattern tops
// out at 3.6-4.4 TB/s on B200 (pcnn_measure_tma_read, mode 2) against 6.7-7.1 TB/s for contiguous boxes -- the kernel sat
// exactly on that ceiling (4.6 TB/s, profiles/r01_README.md).  Here every TMA box is a contiguous run of one dy row:
//   (More than 64 filters: K/64 channel groups per dy row -- K/64 x 4 boxes per stage and K/64 x 4 MMAs per row; K <= 256.)
//   * A CTA owns a strip of <= 120 output columns and walks DOWN the rows of its share of the images.  One dy row of the
//     strip is an A operand [128 pixels x 64 channels] (4 boxes of <= 32 pixels, one per TMEM lane quarter, overlapping by
//     S-1 pixels so that the shift along s never crosses a warp).
//   * The accumulator is a RING OF OUTPUT ROWS in TMEM: slot t holds dx row t of the walk as SCP = 4*ceil(S*C/4) columns
//     (s, c).  dy row p contributes to rows p .. p+R-1, i.e. to R consecutive slots = one window of R*SCP columns, so the sum
//     over r is done by the tensor core (4 MMAs M=128, N=48, K=16 per dy row against a constant 6 KB filter matrix whose
//     columns are (r, s, c)) and the window slides by one slot per row.  Row t is complete once dy row t has been added; it
//     is then drained by the epilogue (sum over s = a shuffle across lanes, bf16, coalesced store) and re-zeroed.
//   * Flow control is per group of 8 slots (tcgen05.commit -> tfull, epilogue -> tempty), NG groups in flight.
//   * A CTA's share starts mid-image in general: the R-1 rows above it are replayed with filter variants that keep only the
//     contributions landing inside the share (0.5 % extra reads at config 5).
//   * Window step st > 1 (template parameter ST): the walk still covers every dx row; dy row h/st enters the ring at the slot of
//     dx row h when h % st == 0.  A lane holds one dy pixel and owns the st dx columns (pixel + M - 1) * st + phi, M = ceil(S/st),
//     phi < st: each is a sum over m of column (phi + m*st, c) of the lane m below it, so the boxes overlap by M - 1 pixels.
//     Rows and columns no tap reaches come out as zeros.
// TMEM addressing: the accumulator window of a tcgen05.mma must start on a multiple of 4 columns (an arbitrary column faults
// with "misaligned address" on B200), hence SCP = 4*ceil(S*C/4) columns per slot.
// Issue budget (pcnn_measure_mma_rate): one tcgen05.mma of N <= 112 occupies the issue/tensor path ~56-70 clk whatever its
// size, so 4 MMAs per 15 KB of dy fit under the ~630 clk of HBM time those bytes cost one SM.
#include "tc_common.cuh"

#include <stdlib.h>

using namespace pcnn_tc;

namespace {

constexpr int D2_THREADS = 192;          // warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue (lane quarters)
constexpr int D2_HALF_BYTES = 16384;     // one group of 64 channels: 4 quarters x 32 pixel rows x 128 B
constexpr int D2_MAX_STAGES = 11;
constexpr int D2_MAX_NG = 6;
constexpr int D2_GROUP = 8;
constexpr int D2_SMEM_BUDGET = 200 * 1024;

struct Dgrad2Params {
    int n_img, H, W, P, Q;
    int nstrips, strip_w, oq, bp;        // strips per row, output columns per strip, dy pixels per lane quarter / per TMA box
    int ng, ring, stages;                // slot groups in flight, ring slots (8 * ng), smem stages
    int KH;                              // channels / 64: a TMA box holds 64 channels (one 128-byte swizzle row per pixel)
    long long T;                         // n_img * H output rows in walk order
    long long dx_pitch, dx_image_rows;
    __nv_bfloat16 *dx;
};

struct Dgrad2Ctl {
    unsigned long long full[D2_MAX_STAGES], empty[D2_MAX_STAGES], tfull[D2_MAX_NG], tempty[D2_MAX_NG], bfull;
    uint32_t tmem_base;
};

// F_v[n][k] for window column n = r' * SCP + s * C + c: f[k][r' + v][s][c] (variant v drops the first v filter rows), zero padding
// layout [variant][channel group of 64][nw][64]
__global__ void k_dgrad2_build_variants(const float *__restrict__ f, __nv_bfloat16 *__restrict__ T, int nw, int scp, int K, int R, int S,
                                        int C) {
    const int total = R * nw * K, KH = K / 64;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int kl = idx % 64, n = (idx / 64) % nw, kh = (idx / (64 * nw)) % KH, v = idx / (64 * nw * KH), k = kh * 64 + kl;
        const int r = n / scp + v, j = n % scp;
        float val = 0.0f;
        if (r < R && j < S * C) val = f[(((long)k * R + r) * S + j / C) * C + j % C];
        T[idx] = __float2bfloat16_rn(val);
    }
}

// the rows one CTA feeds to the tensor core, in order: R-1 replayed rows above its share, then its own rows
struct RowWalk {
    long long t0, t1;       // share [t0, t1) of the walk
    int H, P;
    __device__ RowWalk(const Dgrad2Params &p, int idx, int cnt) : H(p.H), P(p.P) {
        const long long L = (p.T + cnt - 1) / cnt;
        t0 = (long long)idx * L;
        t1 = t0 + L < p.T ? t0 + L : p.T;
        if (t0 > t1) t0 = t1;
    }
};

template <int R, int S, int C, int KHC, int ST>
__global__ void __launch_bounds__(D2_THREADS, 1)
k_conv_tc_dgrad_rows(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_b, const Dgrad2Params p) {
    constexpr int SC = S * C, SCP = (SC + 3) / 4 * 4, NW = (R * SCP + 15) / 16 * 16;
    constexpr int M = (S + ST - 1) / ST;                               // dy pixels that reach one dx column
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *base = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    constexpr int BMAT = NW * 128;
    // KHC > 0: the channel-group count is a compile-time constant (64 filters: KHC = 1 keeps the single issuing thread's loop
    // free of the group bookkeeping -- the runtime loop cost 146 -> 187 us at config 5); KHC = 0: p.KH groups at run time
    const int KH = KHC > 0 ? KHC : p.KH, STAGE = KH * D2_HALF_BYTES;
    unsigned char *bvar = base;                                         // [R][KH][NW][64] bf16, SWIZZLE_128B
    unsigned char *astage = base + (size_t)R * KH * BMAT;               // [stages][KH][4][32][64] bf16, SWIZZLE_128B
    Dgrad2Ctl &B = *reinterpret_cast<Dgrad2Ctl *>(astage + (size_t)p.stages * STAGE);
    const int NST = p.stages, NG = p.ng, RING = p.ring;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // this CTA's strip of output columns and its share of the row walk
    const int strip = blockIdx.x % p.nstrips, idx = blockIdx.x / p.nstrips;
    const int cnt = ((int)gridDim.x - strip + p.nstrips - 1) / p.nstrips;
    const RowWalk walk(p, idx, cnt);
    const int w_strip = strip * p.strip_w;
    const int w_end = w_strip + p.strip_w < p.W ? w_strip + p.strip_w : p.W;
    const long long nel = walk.t1 - walk.t0;
    const int h_first = (int)(walk.t0 % p.H);
    const int n_first = (int)(walk.t0 / p.H);
    const int warm = h_first < R - 1 ? h_first : R - 1;               // replayed rows above the share (same image)

    if (threadIdx.x == 0) {
        for (int i = 0; i < NST; ++i) { bar_init(&B.full[i], 1); bar_init(&B.empty[i], 1); }
        for (int i = 0; i < NG; ++i) { bar_init(&B.tfull[i], 1); bar_init(&B.tempty[i], 4); }
        bar_init(&B.bfull, 1);
        fence_barrier_init();
    }
    // pixel rows a box does not cover (box of bp < 32 pixels) must hold finite values: their TMEM lanes are never read
    for (int i = threadIdx.x * 16; i < NST * STAGE; i += D2_THREADS * 16) *reinterpret_cast<uint4 *>(astage + i) = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    if (warp == 1) tc_alloc(&B.tmem_base, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = B.tmem_base;
    if (warp >= 2) {   // every MMA accumulates: the whole ring starts at zero
        const uint32_t t0 = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll
        for (int ch = 0; ch < 16; ++ch) tc_st_zero_32x32(t0 + ch * 32);
        tc_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0 && nel > 0) {
            bar_expect_tx(&B.bfull, (unsigned)(R * KH * BMAT));
            for (int v = 0; v < R * KH; ++v) tma_load_2d(bvar + (size_t)v * BMAT, &map_b, 0, v * NW, &B.bfull);
            int stage = 0;
            unsigned ph = 0;
            int n = n_first, h = h_first - warm;
            const long long nrows = nel + warm;
            for (long long i = 0; i < nrows; ++i) {
                if (h % ST == 0 && h / ST < p.P) {     // dy row h / st enters at dx row h
                    bar_wait_relaxed(&B.empty[stage], ph ^ 1u, 32);
                    bar_expect_tx(&B.full[stage], (unsigned)(KH * 4 * p.bp * 128));
                    unsigned char *a = astage + (size_t)stage * STAGE;
                    const int row = n * p.P + h / ST;
                    for (int kh = 0; kh < KH; ++kh)
#pragma unroll
                        for (int g = 0; g < 4; ++g)      // pixels left of the image / right of its last dy pixel arrive as zeros
                            tma_load_3d(a + kh * D2_HALF_BYTES + g * 4096, &map_dy, kh * 64, w_strip / ST + g * p.oq - (M - 1), row, &B.full[stage]);
                    if (++stage == NST) { stage = 0; ph ^= 1u; }
                }
                if (++h == p.H) { h = 0; ++n; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0 && nel > 0) {
            const uint32_t idesc = umma_idesc_bf16(128, NW);
            const uint64_t adesc0 = umma_desc_k_sw128(s_u32(astage)), bdesc0 = umma_desc_k_sw128(s_u32(bvar));
            bar_wait(&B.bfull, 0);
            int stage = 0;
            unsigned ph = 0;
            int h = h_first - warm;
            int pos = 0;                                   // ring slot of the current element
            int G = 0, ing = 0;                            // group index, elements done in it
            const long long nrows = nel + warm;
            for (long long i = 0; i < nrows; ++i) {
                const bool warmrow = i < warm;
                if (!warmrow && ing == 0 && G + 1 >= NG) {
                    // the windows of group G reach into ring group (G + 1) % NG: its previous occupant must be drained
                    const int rg = (G + 1) % NG;
                    bar_wait(&B.tempty[rg], (unsigned)(((G + 1) / NG - 1) & 1));
                    tc_fence_after();
                }
                if (h % ST == 0 && h / ST < p.P) {
                    bar_wait(&B.full[stage], ph);
                    tc_fence_after();
                    uint64_t ad = adesc0 + (uint64_t)((uint32_t)stage * ((uint32_t)STAGE >> 4));
                    uint64_t bd = bdesc0 + (uint64_t)((uint32_t)(warmrow ? warm - (int)i : 0) * ((uint32_t)(KH * BMAT) >> 4));
                    const uint32_t dcol = tmem + (uint32_t)(pos * SCP);
                    for (int kh = 0; kh < KH; ++kh) {          // 64 channels = 4 K steps of 16
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) tc_mma_bf16(dcol, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc, 1u);
                        ad += D2_HALF_BYTES >> 4;
                        bd += BMAT >> 4;
                    }
                    tc_commit(&B.empty[stage]);
                    if (++stage == NST) { stage = 0; ph ^= 1u; }
                }
                if (++h == p.H) h = 0;
                if (!warmrow) {
                    if (++ing == D2_GROUP || i == nrows - 1) {
                        tc_commit(&B.tfull[G % NG]);
                        ++G;
                        ing = 0;
                    }
                    if (++pos == RING) pos = 0;
                }
            }
        }
    } else {
        // ===== epilogue: drain completed rows, sum over s across lanes, store, re-zero =====
        const int quarter = warp & 3;
        const uint32_t tq = tmem + ((uint32_t)(quarter * 32) << 16);
        const int w_q0 = w_strip + quarter * p.oq * ST;
        int nvalid = w_end - w_q0;                           // output columns of this quarter
        if (nvalid > p.oq * ST) nvalid = p.oq * ST;
        int n = n_first, h = h_first, pos = 0;
        const int ngroups = (int)((nel + D2_GROUP - 1) / D2_GROUP);
        for (int G = 0; G < ngroups; ++G) {
            bar_wait_relaxed(&B.tfull[G % NG], (unsigned)((G / NG) & 1), 64);
            tc_fence_after();
            long long left = nel - (long long)G * D2_GROUP;
            const int nsl = left < D2_GROUP ? (int)left : D2_GROUP;
            for (int i = 0; i < nsl; ++i) {
                uint32_t v[SCP], u[SCP];
                const uint32_t c0 = tq + (uint32_t)(pos * SCP);
#pragma unroll
                for (int j = 0; j < SCP; j += 4) tc_ld_32x4(c0 + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
                const bool tail = pos < R - 1;               // rows written past the ring end by the previous lap
                if (tail) {
#pragma unroll
                    for (int j = 0; j < SCP; j += 4) tc_ld_32x4(tq + (uint32_t)((RING + pos) * SCP) + j, u[j], u[j + 1], u[j + 2], u[j + 3]);
                }
                tc_wait_ld();
                float o[ST * C];
#pragma unroll
                for (int c = 0; c < ST * C; ++c) o[c] = 0.0f;
#pragma unroll
                for (int m = 0; m < M; ++m) {
#pragma unroll
                    for (int phi = 0; phi < ST; ++phi) {
                        const int s = phi + m * ST;
                        if (s >= S) continue;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            float x = __uint_as_float(v[s * C + c]);
                            if (tail) x += __uint_as_float(u[s * C + c]);
                            // lane l holds dy pixel (first + l); its dx columns (first + l + M-1) * st + phi need dy pixel l + (M-1) - m
                            if (M - 1 - m > 0) x = __shfl_down_sync(0xFFFFFFFFu, x, M - 1 - m);
                            o[phi * C + c] += x;
                        }
                    }
                }
                __nv_bfloat16 *dst = p.dx + ((long long)n * p.dx_image_rows + h) * p.dx_pitch + (long long)(w_q0 + lane * ST) * C;
#pragma unroll
                for (int phi = 0; phi < ST; ++phi)
                    if (lane * ST + phi < nvalid) {
#pragma unroll
                        for (int c = 0; c < C; ++c) dst[phi * C + c] = __float2bfloat16_rn(o[phi * C + c]);
                    }
#pragma unroll
                for (int j = 0; j < SCP; j += 4) tc_st_zero_32x4(c0 + j);
                if (tail) {
#pragma unroll
                    for (int j = 0; j < SCP; j += 4) tc_st_zero_32x4(tq + (uint32_t)((RING + pos) * SCP) + j);
                }
                if (++pos == RING) pos = 0;
                if (++h == p.H) { h = 0; ++n; }
            }
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) bar_arrive(&B.tempty[G % NG]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tc_dealloc(tmem, 512);
    }
}

struct Geometry { int scp, nw, ng; };

Geometry geometry(int R, int S, int C) {
    Geometry g;
    g.scp = (S * C + 3) / 4 * 4;
    g.nw = (R * g.scp + 15) / 16 * 16;
    g.ng = 0;
    while (g.ng < D2_MAX_NG && (D2_GROUP * (g.ng + 1) + R - 1) * g.scp + (g.nw - R * g.scp) <= 512) ++g.ng;
    return g;
}

template <int R, int S, int C, int KHC, int ST>
int launch_rows_k(pcnn_ctx *ctx, const CUtensorMap &map_dy, const CUtensorMap &map_b, const Dgrad2Params &p, int grid, size_t smem) {
    static bool configured[64] = {};        // function attributes are per device
    if (!configured[ctx->device & 63]) {
        PCNN_CUDA(cudaFuncSetAttribute(k_conv_tc_dgrad_rows<R, S, C, KHC, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, D2_SMEM_BUDGET + 2048));
        configured[ctx->device & 63] = true;
    }
    k_conv_tc_dgrad_rows<R, S, C, KHC, ST><<<grid, D2_THREADS, smem, ctx->stream>>>(map_dy, map_b, p);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}
template <int R, int S, int C, int ST>
int launch_rows(pcnn_ctx *ctx, const CUtensorMap &map_dy, const CUtensorMap &map_b, const Dgrad2Params &p, int grid, size_t smem) {
    return p.KH == 1 ? launch_rows_k<R, S, C, 1, ST>(ctx, map_dy, map_b, p, grid, smem) : launch_rows_k<R, S, C, 0, ST>(ctx, map_dy, map_b, p, grid, smem);
}

// the built (R, S, C, stride) combinations, in one place for the predicate and the dispatch: every 3x3 (C in {1,2,3,4,8}), 5x5
// (C in {1,3}) and 7x7 (C = 1) kernel at strides 1 and 2; 3x3 with C in {1,2,3} at stride 3; 3x3x3 and 5x5x1 at stride 4
#define PCNN_DGRAD_ROWS_KERNELS(X)                                                                                               \
    X(3, 3, 3, 1) X(3, 3, 1, 1) X(3, 3, 4, 1) X(5, 5, 1, 1) X(3, 3, 2, 1) X(3, 3, 8, 1) X(5, 5, 3, 1) X(7, 7, 1, 1)            \
    X(3, 3, 3, 2) X(3, 3, 1, 2) X(3, 3, 4, 2) X(5, 5, 1, 2) X(3, 3, 2, 2) X(3, 3, 8, 2) X(5, 5, 3, 2) X(7, 7, 1, 2)            \
    X(3, 3, 1, 3) X(3, 3, 2, 3) X(3, 3, 3, 3)                                                                                   \
    X(3, 3, 3, 4) X(5, 5, 1, 4)

bool instantiated(int R, int S, int C, int st) {
#define X(r, s, c, t) if (R == r && S == s && C == c && st == t) return true;
    PCNN_DGRAD_ROWS_KERNELS(X)
#undef X
    return false;
}

// column strips of a multiple of st dx columns; a lane quarter takes oq dy pixels = oq * st dx columns, at most 32 - (M - 1)
// pixels (its box holds oq + M - 1 <= 32 pixels)
struct Strips { int nstrips, strip_w, oq; };
Strips strips(int W, int S, int st) {
    Strips t;
    const int oq_max = 32 - ((S + st - 1) / st - 1);
    t.nstrips = (W + 4 * oq_max * st - 1) / (4 * oq_max * st);
    t.strip_w = ((W + t.nstrips - 1) / t.nstrips + st - 1) / st * st;
    t.oq = (t.strip_w / st + 3) / 4;
    return t;
}

}  // namespace

bool pcnn_conv_dgrad_rows_ok(int N, int H, int W, int C, int K, int R, int S, int stride, const void *dy) {
    if (K % 64 || K > 256 || ((uintptr_t)dy & 15) || N <= 0 || H < R || W < S) return false;
    if (!instantiated(R, S, C, stride)) return false;
    const Geometry g = geometry(R, S, C);
    return g.ng >= 2 && g.nw <= 256 && S <= 16;
}

// host-side tiling of the row-streaming input gradient, for pcnn_conv_bwd_plan_info (no GPU needed)
void pcnn_conv_dgrad_rows_info(int H, int W, int C, int K, int R, int S, int stride, int *out4) {
    const Geometry g = geometry(R, S, C);
    const Strips t = strips(W, S, stride);
    const size_t stage_bytes = (size_t)(K / 64) * D2_HALF_BYTES;
    const size_t fixed = (size_t)R * (K / 64) * g.nw * 128 + sizeof(Dgrad2Ctl) + 1024;
    int st = stage_bytes ? (int)(((size_t)D2_SMEM_BUDGET - fixed) / stage_bytes) : 0;
    out4[0] = t.nstrips; out4[1] = t.oq * stride; out4[2] = g.ng; out4[3] = st > D2_MAX_STAGES ? D2_MAX_STAGES : st;
    (void)H;
}

// dy_channels: as for pcnn_conv_wgrad_rows (filters dy really holds; the TMA zero-fills the rest of a 64-channel box)
int pcnn_conv_dgrad_rows(pcnn_ctx *ctx, const void *dy_bf16, const float *filt_f32_dev, void *dx_bf16, int N, int H, int W, int C, int K,
                         int R, int S, int stride, int row_pitch, int image_rows, int dy_channels) {
    const uint64_t KD = dy_channels > 0 ? (uint64_t)dy_channels : (uint64_t)K;
    pcnn_device_guard guard(ctx->device);
    const Geometry g = geometry(R, S, C);
    Dgrad2Params p;
    memset(&p, 0, sizeof(p));
    p.n_img = N; p.H = H; p.W = W; p.P = (H - R) / stride + 1; p.Q = (W - S) / stride + 1;
    const Strips t = strips(W, S, stride);
    p.nstrips = t.nstrips;
    p.strip_w = t.strip_w;
    p.oq = t.oq;
    p.bp = p.oq + (S + stride - 1) / stride - 1;
    p.ng = g.ng;
    p.ring = D2_GROUP * g.ng;
    p.T = (long long)N * H;
    p.dx_pitch = row_pitch > 0 ? row_pitch : W * C;
    p.dx_image_rows = image_rows > 0 ? image_rows : H;
    p.dx = reinterpret_cast<__nv_bfloat16 *>(dx_bf16);
    p.KH = K / 64;
    const size_t stage_bytes = (size_t)p.KH * D2_HALF_BYTES;
    const size_t fixed = (size_t)R * p.KH * g.nw * 128 + sizeof(Dgrad2Ctl) + 1024;
    int st = (int)(((size_t)D2_SMEM_BUDGET - fixed) / stage_bytes);
    p.stages = st > D2_MAX_STAGES ? D2_MAX_STAGES : st;
    PCNN_REQUIRE(p.stages >= 2, PCNN_ERR_ARG, "pcnn_conv_dgrad: filter variants leave no room for two stages");
    const size_t smem = fixed + (size_t)p.stages * stage_bytes;

    __nv_bfloat16 *T = nullptr;
    const size_t t_elems = (size_t)R * g.nw * K;
    int rc = pcnn_scratch(ctx, t_elems * 2, (void **)&T);
    if (rc) return rc;
    k_dgrad2_build_variants<<<(int)((t_elems + 255) / 256), 256, 0, ctx->stream>>>(filt_f32_dev, T, g.nw, g.scp, K, R, S, C);
    PCNN_CHECK_LAUNCH(ctx);

    CUtensorMap map_dy, map_b;
    {
        const uint64_t dims[3] = {KD, (uint64_t)p.Q, (uint64_t)N * p.P};
        const uint64_t str[2] = {KD * 2, (uint64_t)p.Q * KD * 2};
        const uint32_t box[3] = {64, (uint32_t)p.bp, 1};
        if ((rc = make_map_bf16(&map_dy, const_cast<void *>(dy_bf16), 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B)))
            return rc;
        const uint64_t bd[2] = {64, (uint64_t)R * p.KH * g.nw};        // [variant][channel group][nw] rows of 64 channels
        const uint64_t bs[1] = {128};
        const uint32_t bb[2] = {64, (uint32_t)g.nw};
        if ((rc = make_map_bf16(&map_b, T, 2, bd, bs, bb, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))) return rc;
    }
    // every CTA needs at least one row of its strip; more CTAs than rows would leave empty shares (handled, but pointless)
    long long want = p.T * p.nstrips;
    const int grid = (int)(want < ctx->sm_count ? want : ctx->sm_count);
#define X(r, s, c, t) if (R == r && S == s && C == c && stride == t) return launch_rows<r, s, c, t>(ctx, map_dy, map_b, p, grid, smem);
    PCNN_DGRAD_ROWS_KERNELS(X)
#undef X
    pcnn_set_error("pcnn_conv_dgrad: no row-streaming instantiation for R = %d, S = %d, C = %d, stride %d", R, S, C, stride);
    return PCNN_ERR_ARG;
}

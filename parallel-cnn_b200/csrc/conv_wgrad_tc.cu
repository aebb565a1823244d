// parallel-cnn_b200/csrc/conv_wgrad_tc.cu -- weight gradient of the NHWC bf16 convolution (64 filters) on the tcgen05 tensor cores.
//
//     dw[k][r][s][c] = sum_{n,p,q} dy[n][p][q][k] * x[n][p*st+r][q*st+s][c]     [ref: layer.h:371-395 bp_weight_c1, without /576]
//
// SURVEY.md x3 / BASELINE.json config 5: dy [N,222,222,64] is 95 % of the 6.6 MB/image this pass moves and the pass is
// HBM-bound (SURVEY.md 8d), so: dy crosses HBM -> shared memory once by TMA and is consumed there by tcgen05.mma.
//   * The reduction runs over pixels, the slow axis of both tensors.  dy needs no transposition: a TMA tile
//     [RB rows][PC pixels][64 filters] is an MN-major B operand as it lands (one 128-byte swizzled row per pixel; the RB
//     rows are RB atoms along N, N = RB * 64 <= 256).
//   * The other operand is the Hankel matrix of the x rows, A[(rho, s, c)][pixel q] = x[p0 + rho][(q + s) * C + c] for the
//     RB + R - 1 input rows a block of RB dy rows touches (54 of M = 64 rows at config 5); eight warps build it in shared
//     memory from the x row segments (x is 5 % of the traffic; the 9x expansion never leaves the SM).
//     Window step st > 1: A[(rho, s, c)][q] = x[p0*st + rho][(q*st + s) * C + c] over the (RB-1)*st + R x rows of the block
//     (the builders gather with a stride of st*C elements); the dy tiles and the MMAs do not change.
//     (More than 64 filters: K/64 boxes per tile, the accumulator columns become (filter group, row, filter), K <= 256.)
//   * D[(rho, s, c)][(row, k)] accumulates in ONE 64 x 256 TMEM accumulator for the whole kernel; the entries with
//     rho - row*st = r in [0, R) are the gradient, the others are discarded.  At the end each CTA folds the RB row blocks,
//     writes one 1,728-float partial, and a second kernel adds the partials in a fixed order (deterministic, no atomics).
// Why this shape: one tcgen05.mma costs the issuing thread and the tensor path ~56-70 clk for any N <= 112 and N/2 clk
// above (pcnn_measure_mma_rate), and a first version with one dy row per tile (dy as the M = 64 operand, N = 32) was bound
// by exactly that: 14 MMAs per 28 KB, 5.2 TB/s with a minimal issue loop, 4.1 TB/s with a careless one, 6.3 TB/s with the
// MMAs removed.  With N = 192 one instruction consumes 6 KB of dy and the kernel streams 6.1 TB/s (92 % of the HBM peak).
#include "tc_common.cuh"

#include <stdlib.h>

using namespace pcnn_tc;

namespace {

constexpr int W2_BUILD_WARPS = 8;
constexpr int W2_THREADS = 64 + 32 * W2_BUILD_WARPS;   // warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-9 Hankel builders
constexpr int W2_MAX_STAGES = 6;
constexpr int W2_ITEMS = 4;                            // 16-byte units of the Hankel tile per builder thread
constexpr int W2_SMEM_BUDGET = 222 * 1024;
constexpr int W2_DUMP_STRIDE = 257;                    // floats per accumulator row in the read-out staging (bank spread)

struct Wgrad2Params {
    int n_img, H, P, Q, W, C, R, SC;
    int RB, NXR, PC, KO;                   // dy rows per tile, x rows per tile, pixels per tile, PC / 8
    int KH;                                // filters / 64: a TMA box (and an MMA atom along N) holds 64 filters
    int nreal, nout;                       // Hankel rows in use (NXR * SC), outputs per filter (R * SC)
    int n_pb, n_ch, stages;                // row blocks per image, pixel chunks per row, smem stages
    long long x_pitch, x_image_rows;
    int xseg_bytes, xseg_stride, xrow_bytes;   // bytes wanted per x segment, smem stride, copyable bytes per x row
    int guard;                             // 1: the copied rows carry pad elements past W*C that must read as zero
    const __nv_bfloat16 *x;
    float *slots;                          // [grid][64 * nout]
};

struct Wgrad2Ctl {
    unsigned long long full[W2_MAX_STAGES], empty[W2_MAX_STAGES], bready[W2_MAX_STAGES], tdone;
    uint32_t tmem_base;
};

__device__ __forceinline__ unsigned short lds_u16(uint32_t saddr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts_v4(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// bytes of x row segment `chunk` that exist in the row (a multiple of 16; 0 when the chunk starts past the row)
template <int ST>
__device__ __forceinline__ int xseg_copy_bytes(const Wgrad2Params &p, int chunk) {
    const int start = chunk * p.PC * ST * p.C * 2;
    int avail = p.xrow_bytes - start;
    if (avail < 0) avail = 0;
    return avail < p.xseg_bytes ? avail : p.xseg_bytes;
}

// CT = compile-time input-channel count (the gather stride of the Hankel builder), 0 = run-time; ST = window step
template <int CT, int ST>
__global__ void __launch_bounds__(W2_THREADS, 1)
k_conv_tc_wgrad_rows(const __grid_constant__ CUtensorMap map_dy, const Wgrad2Params p) {
    const int C = CT > 0 ? CT : p.C;
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *base = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    const int dy_half = p.RB * p.PC * 128;              // one box: [RB][PC][64] bf16, SWIZZLE_128B
    const int dy_bytes = p.KH * dy_half;                // [KH filter groups][RB][PC][64]
    const int ncols = p.KH * p.RB * 64;                 // accumulator columns (group, row, filter)
    const int hk_bytes = 64 * p.PC * 2;                 // Hankel tile [64][PC] bf16, K-major 8x8 core matrices
    const int x_bytes = p.NXR * p.xseg_stride;
    unsigned char *DY = base;
    unsigned char *HK = DY + (size_t)p.stages * dy_bytes;
    unsigned char *X = HK + (size_t)p.stages * hk_bytes;
    Wgrad2Ctl &S = *reinterpret_cast<Wgrad2Ctl *>(X + (size_t)p.stages * x_bytes);
    const int NST = p.stages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_per_img = p.n_pb * p.n_ch;
    const int ntiles = p.n_img * tiles_per_img;
    const int SBO = p.KO * 128;                         // bytes between 8-row groups of the Hankel tile
    const int tmem_cols = ncols <= 64 ? 64 : (ncols <= 128 ? 128 : 256);

    if (threadIdx.x == 0) {
        for (int i = 0; i < NST; ++i) { bar_init(&S.full[i], 1); bar_init(&S.empty[i], 1); bar_init(&S.bready[i], W2_BUILD_WARPS); }
        bar_init(&S.tdone, 1);
        fence_barrier_init();
    }
    // Hankel rows >= nreal and everything the x copies do not reach stay zero / finite for the whole kernel
    for (int i = threadIdx.x * 16; i < NST * (hk_bytes + x_bytes); i += W2_THREADS * 16) *reinterpret_cast<uint4 *>(HK + i) = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    if (warp == 1) tc_alloc(&S.tmem_base, (unsigned)tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S.tmem_base;

    if (warp == 0) {
        // ===== TMA producer: one dy box [64 filters x PC pixels x RB rows] and NXR x row segments per tile =====
        if (lane == 0) {
            int stage = 0;
            unsigned ph = 0;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int n = tile / tiles_per_img, rem = tile % tiles_per_img, pb = rem / p.n_ch, ch = rem % p.n_ch;
                const int p0 = pb * p.RB;
                const int xb = xseg_copy_bytes<ST>(p, ch);
                int nx = p.H - p0 * ST;                   // x rows p0*st .. p0*st + NXR - 1 that exist
                if (nx > p.NXR) nx = p.NXR;
                bar_wait_relaxed(&S.empty[stage], ph ^ 1u, 32);
                bar_expect_tx(&S.full[stage], (unsigned)(dy_bytes + nx * xb));
                for (int kh = 0; kh < p.KH; ++kh)                                             // rows >= P, pixels >= Q: zeros
                    tma_load_4d(DY + (size_t)stage * dy_bytes + (size_t)kh * dy_half, &map_dy, kh * 64, ch * p.PC, p0, n, &S.full[stage]);
                if (xb > 0)
                    for (int r = 0; r < nx; ++r)
                        tma_load_1d(X + (size_t)stage * x_bytes + (size_t)r * p.xseg_stride,
                                    p.x + ((long long)n * p.x_image_rows + p0 * ST + r) * p.x_pitch + (long long)ch * p.PC * ST * C, (unsigned)xb,
                                    &S.full[stage]);
                if (++stage == NST) { stage = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: D[64 x RB*64] += Hankel[64 x 16 pixels] * dy[16 pixels x RB*64]; invariant operands, constant adds =====
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_bf16(64, ncols, /*A K-major*/ 0, /*B MN-major*/ 1);
            const uint64_t adesc0 = umma_desc_k_none(s_u32(HK), 128, (uint32_t)SBO);
            const uint64_t bdesc0 = umma_desc(s_u32(DY), (uint32_t)(p.PC * 128), 1024, 2);   // LBO = next dy row, SBO = next 8 pixels
            const uint32_t a_step = (uint32_t)hk_bytes >> 4, b_step = (uint32_t)dy_bytes >> 4;
            const int nk = p.PC / 16;
            int stage = 0;
            unsigned ph = 0;
            bool first = true;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                bar_wait(&S.full[stage], ph);
                bar_wait(&S.bready[stage], ph);
                tc_fence_after();
                uint64_t ad = adesc0 + (uint64_t)((uint32_t)stage * a_step), bd = bdesc0 + (uint64_t)((uint32_t)stage * b_step);
                tc_mma_bf16(tmem, ad, bd, idesc, first ? 0u : 1u);
                for (int ks = 1; ks < nk; ++ks) {
                    ad += 256 >> 4;                          // 16 pixels of the Hankel tile: two 128-byte core matrices
                    bd += 2048 >> 4;                         // 16 pixels of dy: two 1024-byte swizzle groups
                    tc_mma_bf16(tmem, ad, bd, idesc, 1u);
                }
                first = false;
                tc_commit(&S.empty[stage]);
                if (++stage == NST) { stage = 0; ph ^= 1u; }
            }
            tc_commit(&S.tdone);
        }
    } else {
        // ===== Hankel builders: 16-byte units = 8 pixels of one row (rho, j); shared-memory loads and stores by address =====
        const int b = threadIdx.x - 64;
        const int units = ((p.nreal + 7) / 8) * 8 * p.KO;
        int src_off[W2_ITEMS], dst_off[W2_ITEMS], e0s[W2_ITEMS];
#pragma unroll
        for (int i = 0; i < W2_ITEMS; ++i) {
            const int L = b + i * (32 * W2_BUILD_WARPS);
            src_off[i] = -1; dst_off[i] = 0; e0s[i] = 0;
            if (L < units) {
                const int n8 = L / (p.KO * 8), rem = L % (p.KO * 8), kk = rem >> 3, nl = rem & 7, n = n8 * 8 + nl;
                if (n < p.nreal) {
                    const int rho = n / p.SC, j = n % p.SC;
                    e0s[i] = kk * 8 * ST * C + j;            // element of the x segment feeding pixel 8*kk of the tile
                    src_off[i] = rho * p.xseg_stride + e0s[i] * 2;
                    dst_off[i] = n8 * SBO + kk * 128 + nl * 16;
                }
            }
        }
        const uint32_t x_s = s_u32(X), hk_s = s_u32(HK);
        int stage = 0;
        unsigned ph = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            bar_wait_relaxed(&S.full[stage], ph, 32);
            const uint32_t xs = x_s + (uint32_t)(stage * x_bytes), hs = hk_s + (uint32_t)(stage * hk_bytes);
            unsigned short e[W2_ITEMS][8];
#pragma unroll
            for (int i = 0; i < W2_ITEMS; ++i) {             // all gathers in flight before the first use
                const uint32_t src = xs + (uint32_t)(src_off[i] >= 0 ? src_off[i] : 0);
#pragma unroll
                for (int u = 0; u < 8; ++u) e[i][u] = lds_u16(src + (uint32_t)(u * ST * C * 2));
            }
            int lim0 = 0;
            if (p.guard) lim0 = p.W * C - ((tile % tiles_per_img) % p.n_ch) * p.PC * ST * C;   // row elements at or after the segment start
#pragma unroll
            for (int i = 0; i < W2_ITEMS; ++i) {
                if (src_off[i] >= 0) {
                    if (p.guard) {
#pragma unroll
                        for (int u = 0; u < 8; ++u)
                            if (e0s[i] + u * ST * C >= lim0) e[i][u] = 0;
                    }
                    uint4 o;
                    o.x = e[i][0] | ((uint32_t)e[i][1] << 16); o.y = e[i][2] | ((uint32_t)e[i][3] << 16);
                    o.z = e[i][4] | ((uint32_t)e[i][5] << 16); o.w = e[i][6] | ((uint32_t)e[i][7] << 16);
                    sts_v4(hs + (uint32_t)dst_off[i], o);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) bar_arrive(&S.bready[stage]);
            if (++stage == NST) { stage = 0; ph ^= 1u; }
        }
    }

    // ===== read-out: accumulator -> shared memory, fold the RB row blocks, one partial per CTA =====
    float *dump = reinterpret_cast<float *>(base);      // the stages are free once every MMA has retired
    if (warp >= 2 && warp < 6) {
        bar_wait_relaxed(&S.tdone, 0, 64);
        tc_fence_after();
        const int quarter = warp & 3;                   // an M = 64 accumulator keeps row n in TMEM lane (n / 16) * 32 + n % 16
        const int n = quarter * 16 + lane;
        for (int c0 = 0; c0 < ncols; c0 += 32) {
            uint32_t v[32];
            tc_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c0, v);
            tc_wait_ld();
            if (lane < 16) {
#pragma unroll
                for (int i = 0; i < 32; ++i) dump[n * W2_DUMP_STRIDE + c0 + i] = __uint_as_float(v[i]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    {
        // dw[k][r][j] = sum over row blocks rb of D[(rb * st + r) * SC + j][rb * 64 + k]
        const int K = p.KH * 64;
        float *dst = p.slots + (size_t)blockIdx.x * K * p.nout;
        for (int o = threadIdx.x; o < K * p.nout; o += W2_THREADS) {
            const int k = o / p.nout, rj = o % p.nout, r = rj / p.SC, j = rj % p.SC, kh = k >> 6, kl = k & 63;
            float s = 0.0f;
            for (int rb = 0; rb < p.RB; ++rb) s += dump[((rb * ST + r) * p.SC + j) * W2_DUMP_STRIDE + (kh * p.RB + rb) * 64 + kl];
            dst[o] = s;
        }
    }
    if (warp == 1) {
        tc_fence_after();
        tc_dealloc(tmem, (unsigned)tmem_cols);
    }
}

// dw[o] = sum over CTAs of slots[cta][o]: 8 threads per output add every 8th partial in order, then a fixed tree over the 8
// (deterministic; 32 outputs x 8 slices per block keeps the loads coalesced)
__global__ void __launch_bounds__(256) k_conv_tc_wgrad_rows_reduce(const float *__restrict__ slots, float *__restrict__ dw, int nslots, int nout) {
    __shared__ float part[8][33];
    const int ox = threadIdx.x & 31, sy = threadIdx.x >> 5;
    const int o = blockIdx.x * 32 + ox;
    float s = 0.0f;
    if (o < nout)
        for (int i = sy; i < nslots; i += 8) s += slots[(size_t)i * nout + o];
    part[sy][ox] = s;
    __syncthreads();
    if (sy == 0 && o < nout)
        dw[o] = ((part[0][ox] + part[1][ox]) + (part[2][ox] + part[3][ox])) + ((part[4][ox] + part[5][ox]) + (part[6][ox] + part[7][ox]));
}

struct Plan { int RB, PC, stages; size_t stage_bytes, smem; bool ok; };

// Tile shape: dy rows per tile RB (N = RB * 64) and pixels per tile PC.  Measured at config 5 (profiles/r01_README.md): what
// matters is that the tiles cover the [P x Q] plane with little padding (PC = 112 covers Q = 222 in two chunks: 139-147 us;
// PC = 80 in three: 149-244 us) and that at least three stages fit; RB = 3 (139 us) ~ RB = 2 (141 us) < RB = 4 (147 us, two
// stages).  Window step st: a block of RB dy rows reads (RB - 1) * st + R x rows, a chunk of PC pixels ((PC - 1) * st + S) * C
// elements of each.
Plan plan_for(int P, int Q, int C, int R, int S, int KH, int st) {
    Plan pl;
    memset(&pl, 0, sizeof(pl));
    const int SC = S * C;
    double best = -1.0;
    for (int RB = 4; RB >= 1; --RB) {
        const int NXR = (RB - 1) * st + R;
        if (NXR * SC > 64 || RB * KH * 64 > 256) continue;
        for (int PC = 128; PC >= 32; PC -= 16) {
            const int units = ((NXR * SC + 7) / 8) * 8 * (PC / 8);
            if (units > W2_ITEMS * 32 * W2_BUILD_WARPS) continue;
            const size_t xseg = (size_t)((((PC - 1) * st + S + 1) * C * 2 + 127) / 128 * 128);
            const size_t stage = (size_t)KH * RB * PC * 128 + (size_t)64 * PC * 2 + (size_t)NXR * xseg;
            int st = (int)(((size_t)W2_SMEM_BUDGET - sizeof(Wgrad2Ctl) - 1024) / stage);
            if (st > W2_MAX_STAGES) st = W2_MAX_STAGES;
            if (st < 2) continue;
            if ((size_t)st * stage < (size_t)64 * W2_DUMP_STRIDE * 4) continue;        // the read-out staging reuses the stages
            // padded volume the tiles stream and multiply, +3 % when only double buffering fits, + a nudge towards larger N
            double cost = (double)((P + RB - 1) / RB * RB) * (double)((Q + PC - 1) / PC * PC) * (st < 3 ? 1.03 : 1.0) * (1.0 + 0.001 * (4 - RB));
            if (best < 0.0 || cost < best) {
                best = cost;
                pl.RB = RB; pl.PC = PC; pl.stages = st; pl.stage_bytes = stage;
                pl.smem = (size_t)st * stage + sizeof(Wgrad2Ctl) + 1024;
                pl.ok = true;
            }
        }
    }
    return pl;
}

template <int CT, int ST>
int launch_rows(pcnn_ctx *ctx, const CUtensorMap &map_dy, const Wgrad2Params &p, int grid, size_t smem) {
    static bool configured[64] = {};        // function attributes are per device
    if (!configured[ctx->device & 63]) {
        PCNN_CUDA(cudaFuncSetAttribute(k_conv_tc_wgrad_rows<CT, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, W2_SMEM_BUDGET + 2048));
        configured[ctx->device & 63] = true;
    }
    k_conv_tc_wgrad_rows<CT, ST><<<grid, W2_THREADS, smem, ctx->stream>>>(map_dy, p);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}
template <int ST>
int launch_rows_c(pcnn_ctx *ctx, const CUtensorMap &map_dy, const Wgrad2Params &p, int grid, size_t smem) {
    return p.C == 3 ? launch_rows<3, ST>(ctx, map_dy, p, grid, smem) : p.C == 1 ? launch_rows<1, ST>(ctx, map_dy, p, grid, smem)
         : p.C == 4 ? launch_rows<4, ST>(ctx, map_dy, p, grid, smem) : launch_rows<0, ST>(ctx, map_dy, p, grid, smem);
}

}  // namespace

bool pcnn_conv_wgrad_rows_ok(int N, int H, int W, int C, int K, int R, int S, int stride, int row_pitch, const void *x, const void *dy) {
    if (K % 64 || K > 256 || ((uintptr_t)dy & 15) || ((uintptr_t)x & 15) || row_pitch % 8 || N <= 0 || H < R || W < S) return false;
    if (stride < 1 || stride > 4) return false;
    return plan_for((H - R) / stride + 1, (W - S) / stride + 1, C, R, S, K / 64, stride).ok;
}

// host-side tile choice of the weight gradient, for pcnn_conv_bwd_plan_info (no GPU needed)
void pcnn_conv_wgrad_rows_info(int H, int W, int C, int K, int R, int S, int stride, int *out4) {
    const Plan pl = plan_for((H - R) / stride + 1, (W - S) / stride + 1, C, R, S, K / 64, stride);
    out4[0] = pl.ok ? 1 : 0; out4[1] = pl.RB; out4[2] = pl.PC; out4[3] = pl.stages;
}

// dy_channels: filters dy really holds per pixel (<= K, multiple of 8: 16-byte pixel pitch); the TMA boxes stay 64 channels
// wide and the hardware fills channels dy_channels..63 of a box with zeros, so a 16- or 32-filter gradient needs no padded copy
int pcnn_conv_wgrad_rows(pcnn_ctx *ctx, const void *x_bf16, const void *dy_bf16, float *dw_f32, int N, int H, int W, int C, int K,
                         int R, int S, int stride, int row_pitch, int image_rows, int dy_channels) {
    const uint64_t KD = dy_channels > 0 ? (uint64_t)dy_channels : (uint64_t)K;
    pcnn_device_guard g(ctx->device);
    const int P = (H - R) / stride + 1, Q = (W - S) / stride + 1;
    const Plan pl = plan_for(P, Q, C, R, S, K / 64, stride);
    PCNN_REQUIRE(pl.ok, PCNN_ERR_ARG, "pcnn_conv_wgrad: shape does not fit the tensor-core kernel");
    Wgrad2Params p;
    memset(&p, 0, sizeof(p));
    p.n_img = N; p.H = H; p.P = P; p.Q = Q; p.W = W; p.C = C; p.R = R; p.SC = S * C;
    p.RB = pl.RB; p.NXR = (pl.RB - 1) * stride + R; p.PC = pl.PC; p.KO = pl.PC / 8; p.KH = K / 64;
    p.nreal = p.NXR * p.SC; p.nout = R * p.SC;
    p.n_pb = (P + p.RB - 1) / p.RB; p.n_ch = (Q + p.PC - 1) / p.PC; p.stages = pl.stages;
    p.x_pitch = row_pitch > 0 ? row_pitch : W * C;
    p.x_image_rows = image_rows > 0 ? image_rows : H;
    p.xseg_bytes = (((p.PC - 1) * stride + S) * C * 2 + 15) / 16 * 16;
    p.xseg_stride = ((((p.PC - 1) * stride + S + 1) * C * 2 + 127) / 128 * 128);
    p.xrow_bytes = (W * C * 2 + 15) / 16 * 16;
    PCNN_REQUIRE((long long)p.xrow_bytes <= p.x_pitch * 2 && p.xseg_bytes <= p.xseg_stride, PCNN_ERR_ARG, "pcnn_conv_wgrad: row pitch");
    p.guard = (W * C * 2) % 16 != 0;
    p.x = reinterpret_cast<const __nv_bfloat16 *>(x_bf16);
    const long ntiles = (long)N * p.n_pb * p.n_ch;
    const int grid = (int)(ntiles < ctx->sm_count ? ntiles : ctx->sm_count);
    const int nout = K * p.nout;
    int rc = pcnn_scratch(ctx, (size_t)grid * nout * sizeof(float), (void **)&p.slots);
    if (rc) return rc;
    CUtensorMap map_dy;
    {
        const uint64_t dims[4] = {KD, (uint64_t)Q, (uint64_t)P, (uint64_t)N};
        const uint64_t str[3] = {KD * 2, (uint64_t)Q * KD * 2, (uint64_t)P * Q * KD * 2};
        const uint32_t box[4] = {64, (uint32_t)p.PC, (uint32_t)p.RB, 1};
        if ((rc = make_map_bf16(&map_dy, const_cast<void *>(dy_bf16), 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B)))
            return rc;
    }
    rc = stride == 1 ? launch_rows_c<1>(ctx, map_dy, p, grid, pl.smem) : stride == 2 ? launch_rows_c<2>(ctx, map_dy, p, grid, pl.smem)
       : stride == 3 ? launch_rows_c<3>(ctx, map_dy, p, grid, pl.smem) : launch_rows_c<4>(ctx, map_dy, p, grid, pl.smem);
    if (rc) return rc;
    k_conv_tc_wgrad_rows_reduce<<<(nout + 31) / 32, 256, 0, ctx->stream>>>(p.slots, dw_f32, grid, nout);
    PCNN_CHECK_LAUNCH(ctx);
    return PCNN_OK;
}

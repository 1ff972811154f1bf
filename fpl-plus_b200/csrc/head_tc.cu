// Tensor-core forward of the network's output conv, nn.Conv3d(ft0 -> classes, k(1,3,3), p(0,1,1))
// (PyMIC/pymic/net/net3d/unet2d5_dsbn.py:268, 306).  With 2..7 classes the direct form is 288 FMAs per voxel on the CUDA
// cores (head_fwd_kernel: FMA-issue bound at 3.5x its HBM time, 53 us at 4x32x128x128) and an implicit GEMM with N = classes
// pays a full 40-cycle MMA per tap for 2 useful columns.  Here the ROW taps are gathered by the tensor pipe and the COLUMN
// taps are scattered over N:
//     Q[v][term, kw, cls] = sum_kh sum_ci x[v + (kh-1) rows][ci] * W_term[cls][ci][kh][kw]     3 * Cin/16 MMAs (A shifted by rows)
//     logits[u][cls]     = bias[cls] + sum_term ( Q[u-1][term,0,cls] + Q[u][term,1,cls] + Q[u+1][term,2,cls] )
//   * the weights stay fp32-accurate: W = W_0 + W_1 + W_2 (three bf16 terms) are three column blocks of B, summed in registers;
//   * input tile = 18 rows x 32 voxels of one plane (one TMA box; rows are exactly four 128-byte core matrices, so any
//     4-row window of the tile is ONE uniform-stride K-major operand); an M tile = 4 rows = 4 warps' worth of TMEM lanes, a
//     WARP = one row: the column taps are two warp shuffles, no shared memory and no block barrier in the epilogue;
//   * output = 16 rows x the 30 interior columns; fp32 NCDHW stores of 30 consecutive floats per warp and class;
//   * warp 0 TMA producer, warp 1 MMA issuer (fully unrolled: 12 / 24 MMAs per tile, two TMEM accumulator sets),
//     warps 2..9 epilogue (two per TMEM lane quarter).
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kHtOutRows = 16, kHtRows = kHtOutRows + 2, kHtCols = 32;     // output rows; input tile
constexpr int kHtOutCols = kHtCols - 2;
constexpr int kHtPlane = kHtRows * kHtCols * 16;           // bytes of one channel group of the tile: 9216
constexpr int kHtEpiWarps = 8;                            // two per TMEM lane quarter
constexpr int kHtThreads = 64 + 32 * kHtEpiWarps;
constexpr int kHtMaxStages = 6;

struct HtParams {
    const float* w;            // [classes][cin][1][3][3]
    const float* bias;
    float* logits;             // [N][classes][D][H][W]
    int N, D, H, W, cin, classes;
    int x_c8off;
    int nb;                    // UMMA N: 9 * classes rounded up to 16
    int a_bytes, stages;
    int mstride, tmem_cols;    // accumulator columns per M tile (32 when nb <= 32: two CTAs per SM), TMEM allocation
    int tiles_h, tiles_w, total_tiles;
};

__device__ __forceinline__ void tmem_ld2(uint32_t taddr, uint32_t& a, uint32_t& b) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "r"(taddr));
}

template <int KSTEPS>      // Cin / 16: the MMA loop is fully unrolled (12 / 24 tiny MMAs per tile: loop control per MMA made the
                           // issuing warp the limit, 2.2 k cycles per tile for 0.5 k of MMAs)
__global__ void __launch_bounds__(kHtThreads) head_fwd_tc_kernel(const __grid_constant__ CUtensorMap xmap, HtParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    // [A stage ring][B: 3 row taps x cin/8 groups x nb x 16 B][barriers]
    uint8_t* ring = smem;
    uint8_t* b_sm = ring + (size_t)P.stages * P.a_bytes;
    const int b_bytes = 3 * (P.cin / 8) * P.nb * 16;
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_sm + ((b_bytes + 127) / 128) * 128);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kHtMaxStages;
    uint64_t* tmem_full = bars + 2 * kHtMaxStages;
    uint64_t* tmem_empty = bars + 2 * kHtMaxStages + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kHtMaxStages + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&xmap) : "memory");
        for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], kHtEpiWarps); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);   // 2 accumulator sets x 4 M tiles x mstride columns
    FPL_PDL_WAIT();
    // B operand (K-major, no swizzle): [kh][k8][n][8 ci] bf16; n = (term * 3 + kw) * classes + cls; K step (kh, j) = 16 channels
    {
        const int groups = P.cin / 8, total = 3 * groups * P.nb * 8;
        __nv_bfloat16* b = reinterpret_cast<__nv_bfloat16*>(b_sm);
        for (int i = threadIdx.x; i < total; i += kHtThreads) {
            int t = i;
            const int kk = t & 7; t >>= 3;
            const int nn = t % P.nb; t /= P.nb;
            const int g = t % groups;
            const int kh = t / groups;
            float v = 0.0f;
            int term = 0;
            if (nn < 9 * P.classes) {
                term = nn / (3 * P.classes);
                const int rem = nn - term * 3 * P.classes;
                const int kw = rem / P.classes, cls = rem - kw * P.classes;
                v = P.w[((int64_t)cls * P.cin + g * 8 + kk) * 9 + kh * 3 + kw];
            }
            const __nv_bfloat16 b0 = __float2bfloat16_rn(v);
            const float r1 = v - __bfloat162float(b0);
            const __nv_bfloat16 b1 = __float2bfloat16_rn(r1);
            const __nv_bfloat16 b2 = __float2bfloat16_rn(r1 - __bfloat162float(b1));
            b[i] = term == 0 ? b0 : (term == 1 ? b1 : b2);
        }
    }
    fence_proxy_async();                                      // generic-proxy writes of B before the tensor pipe reads them
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
                int r = t;
                const int tw = r % P.tiles_w; r /= P.tiles_w;
                const int th = r % P.tiles_h; r /= P.tiles_h;     // r = n * D + d
                mbar_wait(&empty_bar[stage], phase ^ 1);
                mbar_expect_tx(&full_bar[stage], (uint32_t)P.a_bytes);
                // map {W*8 bf16, H, c8tot, D, N}; halo origin (h0 - 1, w0 - 1); outside the plane: zero fill = "same" padding
                tma_load_5d(ring + (size_t)stage * P.a_bytes, &xmap, &full_bar[stage], (tw * kHtOutCols - 1) * 8, th * kHtOutRows - 1,
                            P.x_c8off, r % P.D, r / P.D);
                if (++stage == P.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // K-major A (LBO = channel-group plane, SBO = 128: the tile's core matrices are contiguous) and B (LBO = nb*16, SBO = 128)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(P.nb >> 3) << 17) | (8u << 24);
        const uint64_t a_hi = make_desc(0, kHtPlane, 128), b_hi = make_desc(0, (uint32_t)P.nb * 16, 128);
        const uint64_t b0 = b_hi + (uint64_t)(smem_u32(b_sm) >> 4);
        const uint64_t b_kstep = (uint64_t)(2 * P.nb);            // 16 channels of B, in 16-byte units
        const uint32_t ring_u = smem_u32(ring) >> 4;
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t a0 = a_hi + (uint64_t)(ring_u + (uint32_t)(((size_t)stage * P.a_bytes) >> 4));
            const uint32_t d_acc = tmem_base + (uint32_t)(acc * 4 * P.mstride);
#pragma unroll
            for (int m = 0; m < 4; ++m) {                         // M tile m = output rows 4m .. 4m+3
#pragma unroll
                for (int kh = 0; kh < 3; ++kh) {                  // A = input rows 4m+kh .. 4m+kh+3 (tile row 0 = output row -1)
#pragma unroll
                    for (int j = 0; j < KSTEPS; ++j) {
                        const uint64_t ad = a0 + (uint64_t)((4 * m + kh) * (kHtCols * 16 / 16) + j * (2 * kHtPlane / 16));
                        const uint64_t bd = b0 + (uint64_t)(kh * KSTEPS + j) * b_kstep;
                        if (leader) umma_bf16(d_acc + (uint32_t)(m * P.mstride), ad, bd, idesc, (kh | j) ? 1u : 0u);
                    }
                }
            }
            if (leader) { umma_commit(&empty_bar[stage]); umma_commit(&tmem_full[acc]); }
            __syncwarp();
            if (++stage == P.stages) { stage = 0; phase ^= 1; }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        FPL_PDL_TRIGGER();
    } else {
        // 8 epilogue warps (a warp alone on its scheduler cannot hide the TMEM latency): warps w and w + 4 share a TMEM lane
        // quarter and split the four M tiles of a tile; a warp = one output row, lane = column of the input tile
        const int quarter = warp & 3, pair = (warp - 2) >> 2;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        const int C = P.classes, nvals = 9 * C;
        const int64_t HW = (int64_t)P.H * P.W;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            int r = t;
            const int tw = r % P.tiles_w; r /= P.tiles_w;
            const int th = r % P.tiles_h; r /= P.tiles_h;
            const int dd = r % P.D, n = r / P.D;
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const int w = tw * kHtOutCols + lane - 1;                       // lanes 0 / 31 are the halo columns
            const bool col_ok = lane >= 1 && lane <= kHtOutCols && w < P.W;
#pragma unroll 1
            for (int m = pair; m < 4; m += 2) {
                const int h = th * kHtOutRows + 4 * m + quarter;
                const uint32_t taddr = lane_base + (uint32_t)((acc * 4 + m) * P.mstride);
                float* out = P.logits + (((int64_t)n * C) * P.D + dd) * HW + (int64_t)h * P.W + w;
                const bool in_bounds = col_ok && h < P.H;
                if (C == 2) {                                              // the shipped configurations
                    uint32_t v[16], v16, v17;
                    tmem_ld16(taddr, v);
                    tmem_ld2(taddr + 16, v16, v17);
                    tmem_ld_wait();
                    // n = (term * 3 + kw) * 2 + cls
                    float q[6];
#pragma unroll
                    for (int i = 0; i < 6; ++i) {
                        const float t2 = i < 4 ? __uint_as_float(v[12 + i]) : __uint_as_float(i == 4 ? v16 : v17);
                        q[i] = __uint_as_float(v[i]) + __uint_as_float(v[6 + i]) + t2;
                    }
#pragma unroll
                    for (int cls = 0; cls < 2; ++cls) {
                        const float left = __shfl_up_sync(0xffffffffu, q[cls], 1);          // Q[u-1][kw=0]
                        const float right = __shfl_down_sync(0xffffffffu, q[4 + cls], 1);   // Q[u+1][kw=2]
                        const float y = __ldg(P.bias + cls) + left + q[2 + cls] + right;
                        if (in_bounds) out[(int64_t)cls * P.D * HW] = y;
                    }
                } else {
                    for (int cls = 0; cls < C; ++cls) {
                        float q[3];
#pragma unroll
                        for (int kw = 0; kw < 3; ++kw) {
                            q[kw] = 0.0f;
                            for (int term = 0; term < 3; ++term) {
                                const int col = (term * 3 + kw) * C + cls;
                                uint32_t a, b;
                                tmem_ld2(taddr + (uint32_t)(col & ~1), a, b);
                                tmem_ld_wait();
                                q[kw] += __uint_as_float((col & 1) ? b : a);
                            }
                        }
                        const float left = __shfl_up_sync(0xffffffffu, q[0], 1);
                        const float right = __shfl_down_sync(0xffffffffu, q[2], 1);
                        const float y = __ldg(P.bias + cls) + left + q[1] + right;
                        if (in_bounds) out[(int64_t)cls * P.D * HW] = y;
                    }
                }
            }
            (void)nvals;
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Tensor-core input gradient of the same conv (autograd of unet2d5_dsbn.py:306) for <= 2 classes:
//     dX[v][ci] = sum_kh  sum_(kw, cls)  dL[v + (1-kh) rows + (1-kw) cols][cls] * W[cls][ci][kh][kw]
// The logit gradient is fp32 NCDHW with 1-2 channels, so the A operand is BUILT in shared memory by 8 builder warps: per
// voxel one 16-byte vector holding the (kw, cls) neighbourhood {dL[w+1], dL[w], dL[w-1]} x classes as bf16 -- an im2col
// over the column taps only -- in two planes, the bf16 value and its residual (hi, lo): together the K = 16 of one MMA.
// The row taps are again shifted 4-row windows of the tile (rows are four contiguous 128-byte core matrices), so an M tile
// takes 3 MMAs of N = Cin.  The builders also write the one-channel-group bf16 copy of dL the weight-gradient kernel reads
// and the bias gradient; 8 epilogue warps convert the accumulators to bf16 C8-planar vectors (512 bytes per warp store).
// Replaces head_dgrad_kernel (288 FMAs per voxel on the CUDA cores, 60 us at 4x32x128x128).
constexpr int kHdBuildWarps = 8, kHdEpiWarps = 8;
constexpr int kHdThreads = 32 * (1 + kHdEpiWarps + kHdBuildWarps);
constexpr int kHdStages = 3;
constexpr int kHdStageBytes = 2 * kHtPlane;                 // hi + lo planes of 18 x 32 vectors

struct HdParams {
    const float* w;            // [classes][cin][1][3][3]
    const float* dlogits;      // [N][classes][D][H][W]
    bf16x8* g;                 // input gradient, C8-planar slice (g_c8tot, g_c8off)
    bf16x8* dl8;               // optional: bf16 copy of dL padded to one channel group
    float* dbias;              // optional: [classes], ACCUMULATED into
    int g_c8tot, g_c8off, dl_c8tot, dl_c8off;
    int N, D, H, W, cin, classes;
    int tiles_h, tiles_w, total_tiles;
};

__global__ void __launch_bounds__(kHdThreads) head_dgrad_tc_kernel(HdParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* ring = smem;                                                   // [stage][hi | lo][18][32][16 B]
    uint8_t* b_sm = ring + kHdStages * kHdStageBytes;                       // [kh][hi | lo group][cin][8] bf16
    const int b_bytes = 3 * 2 * P.cin * 16;
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_sm + ((b_bytes + 127) / 128) * 128);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kHdStages;
    uint64_t* tmem_full = bars + 2 * kHdStages;
    uint64_t* tmem_empty = bars + 2 * kHdStages + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kHdStages + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kHdStages; ++s) { mbar_init(&full_bar[s], kHdBuildWarps); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], kHdEpiWarps); }
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 256u);              // 2 accumulator sets x 4 M tiles x 32 columns
    FPL_PDL_WAIT();
    {   // B[kh][group][ci][j = kw * classes + cls] = bf16(W[cls][ci][kh][kw]), the same for the hi and the lo group
        __nv_bfloat16* b = reinterpret_cast<__nv_bfloat16*>(b_sm);
        const int total = 3 * 2 * P.cin * 8;
        for (int i = threadIdx.x; i < total; i += kHdThreads) {
            int t = i;
            const int j = t & 7; t >>= 3;
            const int ci = t % P.cin; t /= P.cin;
            const int kh = t >> 1;
            float v = 0.0f;
            if (j < 3 * P.classes) {
                const int kw = j / P.classes, cls = j - kw * P.classes;
                v = P.w[((int64_t)cls * P.cin + ci) * 9 + kh * 3 + kw];
            }
            b[i] = __float2bfloat16_rn(v);
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int64_t HW = (int64_t)P.H * P.W;
    const int C = P.classes;

    if (warp == 0) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(P.cin >> 3) << 17) | (8u << 24);
        const uint64_t a_hi = make_desc(0, kHtPlane, 128), b_hi = make_desc(0, (uint32_t)P.cin * 16, 128);
        const uint64_t b0 = b_hi + (uint64_t)(smem_u32(b_sm) >> 4);
        const uint64_t b_kh = (uint64_t)(2 * P.cin);              // one kh = two 8-wide K groups, in 16-byte units
        const uint32_t ring_u = smem_u32(ring) >> 4;
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t a0 = a_hi + (uint64_t)(ring_u + (uint32_t)((stage * kHdStageBytes) >> 4));
            const uint32_t d_acc = tmem_base + (uint32_t)(acc * 128);
#pragma unroll
            for (int m = 0; m < 4; ++m) {                         // output rows 4m .. 4m+3
#pragma unroll
                for (int kh = 0; kh < 3; ++kh) {                  // dL rows (4m + 1 - kh ..) = tile rows 4m + 2 - kh ..
                    const uint64_t ad = a0 + (uint64_t)((4 * m + 2 - kh) * (kHtCols * 16 / 16));
                    if (leader) umma_bf16(d_acc + (uint32_t)(m * 32), ad, b0 + (uint64_t)kh * b_kh, idesc, kh ? 1u : 0u);
                }
            }
            if (leader) { umma_commit(&empty_bar[stage]); umma_commit(&tmem_full[acc]); }
            __syncwarp();
            if (++stage == kHdStages) { stage = 0; phase ^= 1; }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        FPL_PDL_TRIGGER();
    } else if (warp <= kHdEpiWarps) {
        // ===================== epilogue: TMEM -> bf16 C8-planar vectors =====================
        const int quarter = warp & 3, pair = (warp - 1) >> 2;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            int r = t;
            const int tw = r % P.tiles_w; r /= P.tiles_w;
            const int th = r % P.tiles_h; r /= P.tiles_h;           // r = n * D + d
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const int w = tw * kHtCols + lane;
#pragma unroll 1
            for (int m = pair; m < 4; m += 2) {
                const int h = th * kHtOutRows + 4 * m + quarter;
                const bool valid = h < P.H && w < P.W;
                bf16x8* out = P.g + ((int64_t)r * P.g_c8tot + P.g_c8off) * HW + (int64_t)h * P.W + w;
                for (int c0 = 0; c0 < P.cin; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld16(lane_base + (uint32_t)(acc * 128 + m * 32 + c0), v);
                    tmem_ld_wait();
                    float f[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) f[i] = __uint_as_float(v[i]);
                    if (valid) {
                        st_bf16x8(out + (int64_t)(c0 / 8) * HW, f);
                        st_bf16x8(out + (int64_t)(c0 / 8 + 1) * HW, f + 8);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else {
        // ===================== builders: fp32 dL -> (kw, cls) im2col vectors, hi / lo planes =====================
        const int bw = warp - 1 - kHdEpiWarps;                        // 0..7: rows bw, bw + 8, bw + 16 of the 18-row tile
        float bsum0 = 0.0f, bsum1 = 0.0f;
        int stage = 0; uint32_t phase = 0;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            int r = t;
            const int tw = r % P.tiles_w; r /= P.tiles_w;
            const int th = r % P.tiles_h; r /= P.tiles_h;
            const int n = r / P.D, dd = r - n * P.D;
            const int h0 = th * kHtOutRows - 1, w = tw * kHtCols + lane;
            const float* base = P.dlogits + (((int64_t)n * C) * P.D + dd) * HW;
            // all global loads of this warp's rows first (one DRAM latency per tile)
            float c0v[3], c1v[3], e0v[3], e1v[3];                     // centre values (cls 0 / 1) and the edge column of lanes 0 / 31
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int row = bw + 8 * k, h = h0 + row;
                const bool row_ok = row < kHtRows && h >= 0 && h < P.H;
                c0v[k] = c1v[k] = e0v[k] = e1v[k] = 0.0f;
                if (row_ok && w < P.W) {
                    c0v[k] = __ldg(base + (int64_t)h * P.W + w);
                    if (C > 1) c1v[k] = __ldg(base + (int64_t)P.D * HW + (int64_t)h * P.W + w);
                }
                const int we = lane == 0 ? w - 1 : w + 1;              // column outside the tile, needed by lanes 0 and 31 only
                if (row_ok && (lane == 0 || lane == 31) && we >= 0 && we < P.W) {
                    e0v[k] = __ldg(base + (int64_t)h * P.W + we);
                    if (C > 1) e1v[k] = __ldg(base + (int64_t)P.D * HW + (int64_t)h * P.W + we);
                }
            }
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* st_hi = ring + stage * kHdStageBytes;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int row = bw + 8 * k;
                if (row < kHtRows) {                                   // warp-uniform
                    // neighbours of the row through shuffles: column w-1 (kw = 2) and w+1 (kw = 0)
                    float l0 = __shfl_up_sync(0xffffffffu, c0v[k], 1), l1 = __shfl_up_sync(0xffffffffu, c1v[k], 1);
                    float r0 = __shfl_down_sync(0xffffffffu, c0v[k], 1), r1 = __shfl_down_sync(0xffffffffu, c1v[k], 1);
                    if (lane == 0) { l0 = e0v[k]; l1 = e1v[k]; }
                    if (lane == 31) { r0 = e0v[k]; r1 = e1v[k]; }
                    // j = kw * classes + cls; kw = 0 reads column w + 1, kw = 2 column w - 1
                    float vals[8];
                    if (C == 2) { vals[0] = r0; vals[1] = r1; vals[2] = c0v[k]; vals[3] = c1v[k]; vals[4] = l0; vals[5] = l1; vals[6] = vals[7] = 0.0f; }
                    else { vals[0] = r0; vals[1] = c0v[k]; vals[2] = l0; vals[3] = vals[4] = vals[5] = vals[6] = vals[7] = 0.0f; }
                    float lo[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) lo[i] = vals[i] - __bfloat162float(__float2bfloat16_rn(vals[i]));
                    bf16x8* dst = reinterpret_cast<bf16x8*>(st_hi) + row * kHtCols + lane;
                    st_bf16x8(dst, vals);
                    st_bf16x8(dst + kHtPlane / 16, lo);
                    // interior rows: the bf16 copy of dL for the weight gradient and the bias gradient
                    const int h = h0 + row;
                    if (row >= 1 && row <= kHtOutRows && h < P.H && w < P.W) {
                        bsum0 += c0v[k]; bsum1 += c1v[k];
                        if (P.dl8 != nullptr) {
                            float cp[8] = {c0v[k], C > 1 ? c1v[k] : 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
                            st_bf16x8(P.dl8 + ((int64_t)r * P.dl_c8tot + P.dl_c8off) * HW + (int64_t)h * P.W + w, cp);
                        }
                    }
                }
            }
            fence_proxy_async();                                       // generic-proxy stores before the tensor pipe reads them
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[stage]);
            if (++stage == kHdStages) { stage = 0; phase ^= 1; }
        }
        if (P.dbias != nullptr) {
            bsum0 = warp_sum(bsum0); bsum1 = warp_sum(bsum1);
            if (lane == 0) {
                atomicAdd(P.dbias, bsum0);
                if (C > 1) atomicAdd(P.dbias + 1, bsum1);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256u);
    }
}

}  // namespace

bool fpl_head_fwd_tc_eligible(int h, int w, int cin, int classes) {
    return cin % 16 == 0 && cin >= 16 && cin <= 64 && classes >= 1 && classes <= 7 && h >= 4 && w >= 32 && (cin == 16 || cin == 32);     // 9 * classes <= 64 accumulator columns per M tile
}

int fpl_head_fwd_tc_launch(const void* x, int x_c8tot, int x_c8off, const float* w, const float* bias, float* logits, int n, int d,
                           int h, int w_, int cin, int classes, void* stream) {
    HtParams P;
    P.w = w; P.bias = bias; P.logits = logits; P.N = n; P.D = d; P.H = h; P.W = w_; P.cin = cin; P.classes = classes;
    P.x_c8off = x_c8off;
    P.nb = ((9 * classes + 15) / 16) * 16;
    P.a_bytes = (cin / 8) * kHtPlane;
    const int b_bytes = ((3 * (cin / 8) * P.nb * 16 + 127) / 128) * 128;
    P.mstride = P.nb <= 32 ? 32 : 64; P.tmem_cols = 8 * P.mstride;
    // nb <= 32 (<= 3 classes): half the TMEM and <= 100 KB of shared memory, so two CTAs share an SM
    const int budget = P.nb <= 32 ? 100 * 1024 : 160 * 1024;
    P.stages = (budget - b_bytes - 512) / P.a_bytes;
    if (P.stages > kHtMaxStages) P.stages = kHtMaxStages;
    FPL_REQUIRE(P.stages >= 2, "fpl_head_fwd: tensor-core tile does not fit shared memory (cin %d, classes %d)", cin, classes);
    const int smem_bytes = P.stages * P.a_bytes + b_bytes + 256 + 1024;
    P.tiles_h = (h + kHtOutRows - 1) / kHtOutRows; P.tiles_w = (w_ + kHtOutCols - 1) / kHtOutCols;
    const int64_t total = (int64_t)P.tiles_h * P.tiles_w * n * d;
    FPL_REQUIRE(total < (1ll << 30), "fpl_head_fwd: too many tiles");
    P.total_tiles = (int)total;
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "fpl_head_fwd: x must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_head_fwd: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap xmap;
    cuuint64_t gdim[5] = {(cuuint64_t)w_ * 8, (cuuint64_t)h, (cuuint64_t)x_c8tot, (cuuint64_t)d, (cuuint64_t)n};
    cuuint64_t gstr[4] = {(cuuint64_t)w_ * 16, (cuuint64_t)h * w_ * 16, (cuuint64_t)x_c8tot * h * w_ * 16,
                          (cuuint64_t)d * x_c8tot * h * w_ * 16};
    cuuint32_t box[5] = {(cuuint32_t)kHtCols * 8, (cuuint32_t)kHtRows, (cuuint32_t)(cin / 8), 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&xmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_head_fwd: cuTensorMapEncodeTiled failed (%d)", (int)r);
    int grid = (P.nb <= 32 ? 2 : 1) * FPL_NUM_SMS;
    if (grid > P.total_tiles) grid = P.total_tiles;
    if (cin == 16) {
        FPL_CHECK_CUDA(cudaFuncSetAttribute(head_fwd_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        fpl_launch(head_fwd_tc_kernel<1>, grid, kHtThreads, smem_bytes, (cudaStream_t)stream, xmap, P);
    } else {
        FPL_CHECK_CUDA(cudaFuncSetAttribute(head_fwd_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        fpl_launch(head_fwd_tc_kernel<2>, grid, kHtThreads, smem_bytes, (cudaStream_t)stream, xmap, P);
    }
    return 0;
}

bool fpl_head_dgrad_tc_eligible(int h, int w, int cin, int classes) {
    return (cin == 16 || cin == 32) && classes >= 1 && classes <= 2 && h >= 4 && w >= 32;
}

int fpl_head_dgrad_tc_launch(const float* dlogits, const float* w, void* g, int g_c8tot, int g_c8off, void* dl8, int dl_c8tot,
                             int dl_c8off, float* dbias, int n, int d, int h, int w_, int cin, int classes, void* stream) {
    HdParams P;
    P.w = w; P.dlogits = dlogits; P.g = (bf16x8*)g; P.dl8 = (bf16x8*)dl8; P.dbias = dbias;
    P.g_c8tot = g_c8tot; P.g_c8off = g_c8off; P.dl_c8tot = dl_c8tot; P.dl_c8off = dl_c8off;
    P.N = n; P.D = d; P.H = h; P.W = w_; P.cin = cin; P.classes = classes;
    P.tiles_h = (h + kHtOutRows - 1) / kHtOutRows; P.tiles_w = (w_ + kHtCols - 1) / kHtCols;
    const int64_t total = (int64_t)P.tiles_h * P.tiles_w * n * d;
    FPL_REQUIRE(total < (1ll << 30), "fpl_head_dgrad: too many tiles");
    P.total_tiles = (int)total;
    const int smem_bytes = kHdStages * kHdStageBytes + ((3 * 2 * cin * 16 + 127) / 128) * 128 + 256 + 1024;
    int grid = 2 * FPL_NUM_SMS;            // two CTAs per SM (57 KB, 256 TMEM columns each): a builder warp's load latency of one
                                           // tile is covered by the other CTA (52.5 -> 38.2 us at Cin 16)
    if (grid > P.total_tiles) grid = P.total_tiles;
    FPL_CHECK_CUDA(cudaFuncSetAttribute(head_dgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    fpl_launch(head_dgrad_tc_kernel, grid, kHdThreads, smem_bytes, (cudaStream_t)stream, P);
    return 0;
}

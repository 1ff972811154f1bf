// Weight gradient of nn.Conv3d k(3,3,3) "same" for the SMALL-channel layers (Cin 16 / 32: levels 0-1 of the network,
// autograd of PyMIC/pymic/net/net3d/unet2d5_dsbn.py:75,79), "h-stacked" form of conv3d_wgrad_tc_kernel.
//
// Why: a tcgen05.mma with both operands in shared memory costs max((M + N) / 4, N / 2) cycles (tools/umma_feed_probe.cu:
// the 128 B/clk shared-memory port, whatever the layout, swizzle or alignment), so with Cout = 16 the small N of the
// depth-stacked tiles of conv3d_wgrad_tc_kernel (M = 64, N = 32: 30.5 cycles for 6 useful 16x16x16 blocks) leaves the
// kernel at 20 % of the tensor peak.  Here BOTH spatial directions that are not the reduction's K direction are stacked:
//   * the TMA boxes are fetched through tensor maps whose dimensions are ordered (w, c8, d, h, n), so a tile lands as
//     [row][depth plane][channel group][voxel][8 ch]: the (plane, channel group) slabs of consecutive ROWS follow each
//     other at ONE uniform stride (the row pitch), which is what an MN-major UMMA operand needs;
//   * B = dy: N = 64 = (2 rows) x (2 planes) x 16 output channels;
//   * Cin 16: A = x: M = 128 = (2 rows) x (4 planes) x 16 input channels; two MMAs per in-plane column tap kw cover the
//     x rows {2i-1, 2i} and {2i+1, 2i+2} against the dy rows {2i, 2i+1}: 18 of the 32 blocks of an MMA are taps and a K
//     step of 16 voxels x 2 rows x 2 planes takes 6 MMAs of 48 cycles (9 x 30.5 cycles for half the voxels before);
//   * Cin 32: M = 128 = (4 planes) x 32 input channels of ONE row; the four x rows of a dy row pair are four MMAs whose
//     accumulators SLIDE over the columns (column block = row tap kh), the two edge rows with N = 32, so no TMEM column
//     and no MMA column is spent on a block that is not a tap; 12 MMAs (533 cycles) per K step.
//   * K = 16 consecutive voxels of a row; the column taps kw are the same tile through descriptors shifted by 16 bytes.
// Accumulators stay in TMEM over the CTA's whole split-K slice; the epilogue folds the four (dy row, dy plane) blocks of a
// tap in SHARED memory (one phase per block: every (accumulator, lane) is then a different tap, plain read-modify-write)
// and adds the CTA's [27][16][Cin] tile to global memory with coalesced atomics (4x fewer than one per TMEM element).
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kThreadsH = 192;
constexpr int kMaxStagesH = 6;
constexpr int kSmemBudgetH = 220 * 1024;

struct HsParams {
    float* dw;
    int N, D, H, W, cin, cout;
    int x_c8off, dy_c8off;
    int th, tw, G;                 // tile rows (even) / columns (16 or 32); G = cin / 8
    int sx, sdy;                   // byte stride of one (plane, channel group) slab in the x / dy tile = row pitch
    int x_bytes, dy_bytes, dy_off, stage_bytes, stages;
    int tiles_h, tiles_w, dplanes, tiles_total, split, nchunks;
    int tapmajor;
};

__device__ __forceinline__ void tmem_st_zero16_hs(uint32_t taddr) {
    const uint32_t z = 0u;
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};"
        ::"r"(taddr), "r"(z) : "memory");
}

__global__ void __launch_bounds__(kThreadsH) conv3d_wgrad_hs_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                   const __grid_constant__ CUtensorMap dymap, HsParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kMaxStagesH;
    uint64_t* done_bar = bars + 2 * kMaxStagesH;
    uint64_t* zero_bar = bars + 2 * kMaxStagesH + 1;       // accumulators zeroed by the epilogue warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStagesH + 2);
    uint8_t* ring = smem + 256;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slice = blockIdx.x % P.split, nc = blockIdx.x / P.split;
    const int tile_begin = (int)(((int64_t)P.tiles_total * slice) / P.split);
    const int tile_end = (int)(((int64_t)P.tiles_total * (slice + 1)) / P.split);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&xmap) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&dymap) : "memory");
        for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(done_bar, 1);
        mbar_init(zero_bar, 4);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512u);
    FPL_PDL_WAIT();      // prologue above overlapped the previous kernel's tail; from here on its results are visible
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int ncols = P.G == 2 ? 6 * 64 : 3 * 96;           // accumulator columns in use

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int t = tile_begin; t < tile_end; ++t) {
                // depth runs fastest (the two x planes neighbouring depth steps share are re-read by the same SM)
                int r = t;
                const int dp = r % P.dplanes; r /= P.dplanes;
                const int tw_i = r % P.tiles_w; r /= P.tiles_w;
                const int th_i = r % P.tiles_h;
                const int n = r / P.tiles_h;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* x_dst = ring + (size_t)stage * P.stage_bytes;
                mbar_expect_tx(&full_bar[stage], (uint32_t)(P.x_bytes + P.dy_bytes));
                // map dimensions (w in 8-byte units, c8, d, h, n); planes / rows / columns outside the volume: zero fill
                tma_load_5d(x_dst, &xmap, &full_bar[stage], 2 * (tw_i * P.tw - 1), P.x_c8off, 2 * dp - 1, th_i * P.th - 1, n);
                tma_load_5d(x_dst + P.dy_off, &dymap, &full_bar[stage], 2 * (tw_i * P.tw), P.dy_c8off + nc * 2, 2 * dp, th_i * P.th, n);
                if (++stage == P.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: the whole warp runs the loop (uniform), one lane issues =====================
        // kind::f16, bf16 x bf16 -> fp32, A and B both MN-major (bits 15, 16), M = 128
        const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t idesc64 = idesc0 | ((uint32_t)(64 >> 3) << 17), idesc32 = idesc0 | ((uint32_t)(32 >> 3) << 17);
        // LBO = stride of the two 8-voxel core matrices of a K step (contiguous in the row), SBO = slab stride
        const uint64_t a_hi = make_desc(0, 128u, (uint32_t)P.sx), b_hi = make_desc(0, 128u, (uint32_t)P.sdy);
        // All descriptor arithmetic below is 64-bit ADDs of warp-uniform values (the start-address field is the low 14
        // bits and never carries): the compiler keeps it on the uniform datapath, 2-3 instructions per MMA.  Building each
        // descriptor as hi | (uint32 expression) cost ~12 per-thread instructions + R2UR moves per MMA and made the issuing
        // warp, not the tensor pipe, the limit (67-78 cycles per 48-cycle MMA).
        const uint64_t xrow = (uint64_t)((uint32_t)(4 * P.G * P.sx) >> 4), dyrow = (uint64_t)((uint32_t)(4 * P.sdy) >> 4);   // row pitch, 16-byte units
        const uint32_t ring_u = smem_u32(ring);
        const bool leader = elect_one();
        const bool committer = elect_one();
        // per-MMA constants of a K step
        uint64_t a_off[12];
        uint32_t d_col[12];
        if (P.G == 2) {
#pragma unroll
            for (int k = 0; k < 6; ++k) { a_off[k] = (uint64_t)(k & 1) * 2 * xrow + (uint64_t)(k >> 1); d_col[k] = tmem_base + (uint32_t)(k * 64); }
#pragma unroll
            for (int k = 6; k < 12; ++k) { a_off[k] = 0; d_col[k] = 0; }
        } else {
            // x row 2i-1+q (tile row 2i+q) against dy rows {2i, 2i+1}: row tap kh = q - b_h; column block = 2 - kh
            //   q=0: kh 0 of row 2i (N 32, block 2) | q=1: kh 1 | kh 0 (N 64, blocks 1-2) | q=2: kh 2 | kh 1 (N 64, blocks 0-1)
            //   q=3: kh 2 of row 2i+1 (N 32, block 0, B = dy row 2i+1)
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                const int kw = k >> 2, q = k & 3;
                a_off[k] = (uint64_t)q * xrow + (uint64_t)kw;
                d_col[k] = tmem_base + (uint32_t)(kw * 96 + (q == 0 ? 64 : (q == 1 ? 32 : 0)));
            }
        }
        int stage = 0; uint32_t phase = 0;
        mbar_wait(zero_bar, 0);
        tc_fence_after();
        const int nsteps_s = P.tw / 16, nsteps_i = P.th / 2;
        for (int t = tile_begin; t < tile_end; ++t) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t x_u = (ring_u + (uint32_t)stage * (uint32_t)P.stage_bytes) >> 4;
            uint64_t a_i = a_hi + (uint64_t)x_u;
            uint64_t b_i = b_hi + (uint64_t)(x_u + ((uint32_t)P.dy_off >> 4));
            for (int i = 0; i < nsteps_i; ++i) {
                uint64_t a_s = a_i, b_s = b_i;
                for (int s = 0; s < nsteps_s; ++s) {
                    if (P.G == 2) {
#pragma unroll
                        for (int k = 0; k < 6; ++k)
                            if (leader) umma_bf16(d_col[k], a_s + a_off[k], b_s, idesc64, 1u);
                    } else {
                        const uint64_t b_s1 = b_s + dyrow;                                  // dy row 2i+1 alone
#pragma unroll
                        for (int k = 0; k < 12; ++k) {
                            const int q = k & 3;
                            if (leader) umma_bf16(d_col[k], a_s + a_off[k], q == 3 ? b_s1 : b_s, (q == 0 || q == 3) ? idesc32 : idesc64, 1u);
                        }
                    }
                    a_s += 16; b_s += 16;
                }
                a_i += 2 * xrow; b_i += 2 * dyrow;
            }
            if (committer) umma_commit(&empty_bar[stage]);
            __syncwarp();
            if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
        if (committer) umma_commit(done_bar);
        __syncwarp();
        FPL_PDL_TRIGGER();   // this CTA has issued its last tile: the next kernel of the stream may be scheduled as SMs drain
    } else {
        // ===================== epilogue warps: zero the accumulators, then TMEM -> shared fold -> global atomics ========
        const int quarter = warp & 3;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        for (int col = 0; col < ncols; col += 16) tmem_st_zero16_hs(lane_base + (uint32_t)col);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(zero_bar);
        if (tile_end > tile_begin) {
            mbar_wait(done_bar, 0);
            tc_fence_after();
            // every MMA has completed, so every TMA box has landed and been consumed: the stage ring is free
            float* acc_sm = reinterpret_cast<float*>(ring);
            const int et = threadIdx.x - 64;                                   // 0..127
            const int tile_elems = 27 * 16 * P.cin;
            for (int e = et * 4; e < tile_elems; e += 128 * 4) *reinterpret_cast<float4*>(acc_sm + e) = make_float4(0.f, 0.f, 0.f, 0.f);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const int L = quarter * 32 + lane;                                 // TMEM lane = M row
            // The (dy row, dy plane) column blocks of an accumulator are different taps for every lane, but for ONE such
            // block every (accumulator, lane) pair is a different tap: one phase per block, plain read-modify-write.
            if (P.G == 2) {
                const int a = L >> 6, a_d = (L >> 4) & 3, ci = L & 15;
#pragma unroll 1
                for (int ph = 0; ph < 4; ++ph) {
                    const int b_h = ph >> 1, b_d = ph & 1;
                    const int kd = a_d - b_d;
#pragma unroll 1
                    for (int acc = 0; acc < 6; ++acc) {
                        const int kw = acc >> 1, j = acc & 1;
                        const int kh = 2 * j + a - b_h;
                        uint32_t r[16];
                        tmem_ld16(lane_base + (uint32_t)(acc * 64 + ph * 16), r);
                        tmem_ld_wait();
                        if (kh < 0 || kh > 2 || kd < 0 || kd > 2) continue;
                        float* dst = acc_sm + ((kd * 3 + kh) * 3 + kw) * 256 + ci;
#pragma unroll
                        for (int co = 0; co < 16; ++co) dst[co * 16] += __uint_as_float(r[co]);
                    }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
            } else {
                const int a_d = L >> 5, ci = L & 31;
#pragma unroll 1
                for (int b_d = 0; b_d < 2; ++b_d) {
                    const int kd = a_d - b_d;
#pragma unroll 1
                    for (int blk = 0; blk < 9; ++blk) {
                        const int kw = blk / 3, kb = blk - kw * 3, kh = 2 - kb;
                        uint32_t r[16];
                        tmem_ld16(lane_base + (uint32_t)(kw * 96 + kb * 32 + b_d * 16), r);
                        tmem_ld_wait();
                        if (kd < 0 || kd > 2) continue;
                        float* dst = acc_sm + ((kd * 3 + kh) * 3 + kw) * 512 + ci;
#pragma unroll
                        for (int co = 0; co < 16; ++co) dst[co * 32] += __uint_as_float(r[co]);
                    }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
            }
            const int per_tap = 16 * P.cin;
            if (P.tapmajor) {
                // S[tap][cout][cin]: the CTA's 16 output channels are per_tap contiguous floats per tap
                // (starting every slice's walk at another offset, so that concurrent CTAs hit different lines, measured
                // SLOWER: 32 -> 16 97.5 -> 105 us; same-address reductions arriving together combine in L2)
                for (int e = et; e < tile_elems; e += 128) {
                    const int tap = e / per_tap, rem = e - tap * per_tap;
                    atomicAdd(P.dw + ((int64_t)tap * P.cout + nc * 16) * P.cin + rem, acc_sm[e]);
                }
            } else {
                // PyTorch layout [cout][cin][27]
                for (int e = et; e < tile_elems; e += 128) {
                    const int tap = e / per_tap, rem = e - tap * per_tap;
                    const int co = rem / P.cin, ci = rem - co * P.cin;
                    atomicAdd(P.dw + ((int64_t)(nc * 16 + co) * P.cin + ci) * 27 + tap, acc_sm[e]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512u);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Row-stacked weight gradient of the k(1,3,3) HEAD conv (Cin 16, the classes padded to one channel group of 8): no depth
// taps, so the ROWS are stacked instead of the planes.  Tiles land as [plane][row][channel group][voxel] (tensor-map
// dimensions (w, c8, h, d, n)); per K step of 16 voxels one MMA per column tap kw:
//   A = x rows R..R+7 (M = 128 = 8 rows x 16 ci), B = dy rows R..R+5 (N = 48 = 6 rows x 8 co): block (q, b) is row tap
//   kh = q - b, 18 of the 48 blocks are taps; 3 MMAs of 44 cycles per 96 voxels (the plane-stacked form of
//   conv3d_wgrad_tc_kernel: 9 MMAs of 30.5 cycles per 64 voxels, 4 of 16 blocks useful).  The planes of a tile are more K.
struct RsParams {
    float* dw;
    int N, D, H, W, x_c8off, dy_c8off;
    int th, tw, planes;            // tile rows (multiple of 6), columns (16 / 32), planes per tile
    int sx, sdy, x_plane, dy_plane, dy_off, stage_bytes, stages;
    int tiles_h, tiles_w, dsteps, tiles_total, split;
    int tapmajor;
};

__global__ void __launch_bounds__(kThreadsH) conv3d_wgrad_rs_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                   const __grid_constant__ CUtensorMap dymap, RsParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kMaxStagesH;
    uint64_t* done_bar = bars + 2 * kMaxStagesH;
    uint64_t* zero_bar = bars + 2 * kMaxStagesH + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStagesH + 2);
    uint8_t* ring = smem + 256;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slice = blockIdx.x;
    const int tile_begin = (int)(((int64_t)P.tiles_total * slice) / P.split);
    const int tile_end = (int)(((int64_t)P.tiles_total * (slice + 1)) / P.split);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&xmap) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&dymap) : "memory");
        for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(done_bar, 1);
        mbar_init(zero_bar, 4);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 256u);
    FPL_PDL_WAIT();      // prologue above overlapped the previous kernel's tail; from here on its results are visible
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int t = tile_begin; t < tile_end; ++t) {
                int r = t;
                const int dp = r % P.dsteps; r /= P.dsteps;
                const int tw_i = r % P.tiles_w; r /= P.tiles_w;
                const int th_i = r % P.tiles_h;
                const int n = r / P.tiles_h;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* x_dst = ring + (size_t)stage * P.stage_bytes;
                mbar_expect_tx(&full_bar[stage], (uint32_t)(P.planes * (P.x_plane + P.dy_plane)));
                // map dimensions (w in 8-byte units, c8, h, d, n); rows / columns / planes outside the volume: zero fill
                tma_load_5d(x_dst, &xmap, &full_bar[stage], 2 * (tw_i * P.tw - 1), P.x_c8off, th_i * P.th - 1, dp * P.planes, n);
                tma_load_5d(x_dst + P.dy_off, &dymap, &full_bar[stage], 2 * (tw_i * P.tw), P.dy_c8off, th_i * P.th, dp * P.planes, n);
                if (++stage == P.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // kind::f16, bf16 x bf16 -> fp32, A and B MN-major, M = 128, N = 48
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(48 >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
        const uint64_t a_hi = make_desc(0, 128u, (uint32_t)P.sx), b_hi = make_desc(0, 128u, (uint32_t)P.sdy);
        const uint64_t xrow6 = (uint64_t)((uint32_t)(6 * 2 * P.sx) >> 4), dyrow6 = (uint64_t)((uint32_t)(6 * P.sdy) >> 4);
        const uint64_t xpl = (uint64_t)((uint32_t)P.x_plane >> 4), dypl = (uint64_t)((uint32_t)P.dy_plane >> 4);
        const uint32_t ring_u = smem_u32(ring);
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        mbar_wait(zero_bar, 0);
        tc_fence_after();
        const int nsteps_s = P.tw / 16, nsteps_r = P.th / 6;
        for (int t = tile_begin; t < tile_end; ++t) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t x_u = (ring_u + (uint32_t)stage * (uint32_t)P.stage_bytes) >> 4;
            uint64_t a_p = a_hi + (uint64_t)x_u;
            uint64_t b_p = b_hi + (uint64_t)(x_u + ((uint32_t)P.dy_off >> 4));
            for (int p = 0; p < P.planes; ++p, a_p += xpl, b_p += dypl) {
                uint64_t a_r = a_p, b_r = b_p;
                for (int r6 = 0; r6 < nsteps_r; ++r6, a_r += xrow6, b_r += dyrow6) {
                    uint64_t a_s = a_r, b_s = b_r;
                    for (int s = 0; s < nsteps_s; ++s, a_s += 16, b_s += 16) {
#pragma unroll
                        for (int kw = 0; kw < 3; ++kw)
                            if (leader) umma_bf16(tmem_base + (uint32_t)(kw * 48), a_s + (uint64_t)kw, b_s, idesc, 1u);
                    }
                }
            }
            if (leader) umma_commit(&empty_bar[stage]);
            __syncwarp();
            if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
        if (leader) umma_commit(done_bar);
        __syncwarp();
        FPL_PDL_TRIGGER();
    } else {
        const int quarter = warp & 3;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        for (int col = 0; col < 144; col += 16) tmem_st_zero16_hs(lane_base + (uint32_t)col);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(zero_bar);
        if (tile_end > tile_begin) {
            mbar_wait(done_bar, 0);
            tc_fence_after();
            float* acc_sm = reinterpret_cast<float*>(ring);                   // [9 taps][8 co][16 ci]; the ring is free now
            const int et = threadIdx.x - 64;
            for (int e = et; e < 1152; e += 128) acc_sm[e] = 0.0f;
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const int L = quarter * 32 + lane;
            const int q = L >> 4, ci = L & 15;                                 // x row of the stack, input channel
            // one phase per dy row b of the stack: for a fixed b every (lane, kw) is a different tap
#pragma unroll 1
            for (int m = 0; m < 3; ++m) {
                uint32_t r[3][16];
#pragma unroll
                for (int kw = 0; kw < 3; ++kw) tmem_ld16(lane_base + (uint32_t)(kw * 48 + m * 16), r[kw]);
                tmem_ld_wait();
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int kh = q - (2 * m + half);
                    if (kh >= 0 && kh <= 2) {
#pragma unroll
                        for (int kw = 0; kw < 3; ++kw) {
                            float* dst = acc_sm + ((kh * 3 + kw) * 8) * 16 + ci;
#pragma unroll
                            for (int co = 0; co < 8; ++co) dst[co * 16] += __uint_as_float(r[kw][half * 8 + co]);
                        }
                    }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
            }
            for (int e = et; e < 1152; e += 128) {
                if (P.tapmajor) atomicAdd(P.dw + e, acc_sm[e]);            // S[tap][8][16]
                else {
                    const int tap = e >> 7, co = (e >> 4) & 7, c = e & 15;
                    atomicAdd(P.dw + (co * 16 + c) * 9 + tap, acc_sm[e]);   // [8][16][1][3][3]
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256u);
    }
}

// tensor map with dimensions ordered (w [8-byte units], c8, h, d, n): a box lands as [plane][row][channel group][voxel]
CUresult encode_rs(EncodeTiledFn encode, CUtensorMap* map, const void* base, int n, int d, int c8tot, int h, int w, int box_w,
                   int box_c8, int box_h, int box_d) {
    cuuint64_t gdim[5] = {(cuuint64_t)w * 2, (cuuint64_t)c8tot, (cuuint64_t)h, (cuuint64_t)d, (cuuint64_t)n};
    cuuint64_t gstr[4] = {(cuuint64_t)h * w * 16, (cuuint64_t)w * 16, (cuuint64_t)c8tot * h * w * 16,
                          (cuuint64_t)d * c8tot * h * w * 16};
    cuuint32_t box[5] = {(cuuint32_t)box_w * 2, (cuuint32_t)box_c8, (cuuint32_t)box_h, (cuuint32_t)box_d, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// tensor map over the C8-planar activation with dimensions ordered (w [8-byte units], c8, d, h, n): a box lands as
// [row][plane][channel group][voxel]
CUresult encode_hs(EncodeTiledFn encode, CUtensorMap* map, const void* base, int n, int d, int c8tot, int h, int w, int box_w,
                   int box_c8, int box_d, int box_h) {
    cuuint64_t gdim[5] = {(cuuint64_t)w * 2, (cuuint64_t)c8tot, (cuuint64_t)d, (cuuint64_t)h, (cuuint64_t)n};
    cuuint64_t gstr[4] = {(cuuint64_t)h * w * 16, (cuuint64_t)c8tot * h * w * 16, (cuuint64_t)w * 16,
                          (cuuint64_t)d * c8tot * h * w * 16};
    cuuint32_t box[5] = {(cuuint32_t)box_w * 2, (cuuint32_t)box_c8, (cuuint32_t)box_d, (cuuint32_t)box_h, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

}  // namespace

bool fpl_wgrad_hs_eligible(int d, int h, int w, int cin, int cout, int kd, int taps) {
    return kd == 3 && taps == 9 && (cin == 16 || cin == 32) && cout % 16 == 0 && cout > 0 && d >= 2 && h >= 2 && w >= 16;
}

/* returns 0 on launch, > 0 on error (fpl_last_error); the caller has checked fpl_wgrad_hs_eligible */
int fpl_wgrad_hs_launch(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off, float* dw, int n,
                        int d, int h, int w, int cin, int cout, void* stream, int tapmajor) {
    HsParams P;
    P.dw = dw; P.N = n; P.D = d; P.H = h; P.W = w; P.cin = cin; P.cout = cout; P.x_c8off = x_c8off; P.dy_c8off = dy_c8off;
    P.G = cin / 8;
    P.th = h >= 8 ? 8 : ((h + 1) / 2) * 2;
    P.tw = (w >= 32 && P.G == 2) ? 32 : 16;
    P.sx = (P.tw + 2) * 16; P.sdy = P.tw * 16;
    P.x_bytes = (P.th + 2) * 4 * P.G * P.sx;
    P.dy_bytes = P.th * 4 * P.sdy;
    P.dy_off = ((P.x_bytes + 127) / 128) * 128;
    P.stage_bytes = ((P.dy_off + P.dy_bytes + 127) / 128) * 128;
    P.stages = (kSmemBudgetH - 2048) / P.stage_bytes;
    if (P.stages > kMaxStagesH) P.stages = kMaxStagesH;
    FPL_REQUIRE(P.stages >= 2, "fpl_conv3d_wgrad_tc: h-stacked tile does not fit (%d bytes per stage)", P.stage_bytes);
    FPL_REQUIRE(P.stages * P.stage_bytes >= 27 * 16 * cin * 4, "fpl_conv3d_wgrad_tc: epilogue scratch does not fit the stage ring");
    const int smem_bytes = P.stages * P.stage_bytes + 1024 + 256;
    P.tiles_h = (h + P.th - 1) / P.th; P.tiles_w = (w + P.tw - 1) / P.tw; P.dplanes = (d + 1) / 2;
    const int64_t tiles = (int64_t)P.tiles_h * P.tiles_w * P.dplanes * n;
    FPL_REQUIRE(tiles < (1ll << 30), "fpl_conv3d_wgrad_tc: too many tiles");
    P.tiles_total = (int)tiles;
    P.nchunks = cout / 16;
    int split = FPL_NUM_SMS / P.nchunks;
    if (split > P.tiles_total) split = P.tiles_total;
    if (split < 1) split = 1;
    P.split = split;
    P.tapmajor = tapmajor;
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0,
                "fpl_conv3d_wgrad_tc: x/dy must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_conv3d_wgrad_tc: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap xmap, dymap;
    CUresult r = encode_hs(encode, &xmap, x, n, d, x_c8tot, h, w, P.tw + 2, P.G, 4, P.th + 2);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_wgrad_tc: tensor map (x, h-stacked) failed (%d)", (int)r);
    r = encode_hs(encode, &dymap, dy, n, d, dy_c8tot, h, w, P.tw, 2, 2, P.th);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_wgrad_tc: tensor map (dy, h-stacked) failed (%d)", (int)r);
    FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_wgrad_hs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    fpl_launch(conv3d_wgrad_hs_kernel, P.nchunks * split, kThreadsH, smem_bytes, (cudaStream_t)stream, xmap, dymap, P);
    FPL_LAUNCH_CHECK();
    return 0;
}

bool fpl_wgrad_rs_eligible(int d, int h, int w, int cin, int cout, int kd, int taps) {
    return kd == 1 && taps == 9 && cin == 16 && cout == 8 && h >= 6 && w >= 16 && d >= 1;
}

/* k(1,3,3), Cin 16, Cout 8 (the head); dw = S[9][8][16] (tapmajor) or [8][16][1][3][3], ACCUMULATED into */
int fpl_wgrad_rs_launch(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off, float* dw, int n,
                        int d, int h, int w, void* stream, int tapmajor) {
    RsParams P;
    P.dw = dw; P.N = n; P.D = d; P.H = h; P.W = w; P.x_c8off = x_c8off; P.dy_c8off = dy_c8off;
    P.th = h >= 12 ? 12 : 6;
    P.tw = w >= 32 ? 32 : 16;
    P.planes = d >= 2 ? 2 : 1;
    P.sx = (P.tw + 2) * 16; P.sdy = P.tw * 16;
    P.x_plane = (P.th + 2) * 2 * P.sx; P.dy_plane = P.th * P.sdy;
    P.dy_off = ((P.planes * P.x_plane + 127) / 128) * 128;
    P.stage_bytes = ((P.dy_off + P.planes * P.dy_plane + 127) / 128) * 128;
    P.stages = (kSmemBudgetH - 2048) / P.stage_bytes;
    if (P.stages > kMaxStagesH) P.stages = kMaxStagesH;
    FPL_REQUIRE(P.stages >= 2, "fpl_conv3d_wgrad_tc: row-stacked tile does not fit (%d bytes per stage)", P.stage_bytes);
    const int smem_bytes = P.stages * P.stage_bytes + 1024 + 256;
    P.tiles_h = (h + P.th - 1) / P.th; P.tiles_w = (w + P.tw - 1) / P.tw; P.dsteps = (d + P.planes - 1) / P.planes;
    const int64_t tiles = (int64_t)P.tiles_h * P.tiles_w * P.dsteps * n;
    FPL_REQUIRE(tiles < (1ll << 30), "fpl_conv3d_wgrad_tc: too many tiles");
    P.tiles_total = (int)tiles;
    int split = FPL_NUM_SMS;
    if (split > P.tiles_total) split = P.tiles_total;
    P.split = split;
    P.tapmajor = tapmajor;
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0,
                "fpl_conv3d_wgrad_tc: x/dy must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_conv3d_wgrad_tc: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap xmap, dymap;
    CUresult r = encode_rs(encode, &xmap, x, n, d, x_c8tot, h, w, P.tw + 2, 2, P.th + 2, P.planes);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_wgrad_tc: tensor map (x, row-stacked) failed (%d)", (int)r);
    r = encode_rs(encode, &dymap, dy, n, d, dy_c8tot, h, w, P.tw, 1, P.th, P.planes);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_wgrad_tc: tensor map (dy, row-stacked) failed (%d)", (int)r);
    FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_wgrad_rs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    fpl_launch(conv3d_wgrad_rs_kernel, split, kThreadsH, smem_bytes, (cudaStream_t)stream, xmap, dymap, P);
    FPL_LAUNCH_CHECK();
    return 0;
}

// Weight gradient of nn.Conv3d k(kd,3,3) "same" (autograd of PyMIC/pymic/net/net3d/unet2d5_dsbn.py:75,79)
// on the 5th-gen tensor cores:  dW[co][ci][kd][kh][kw] += sum_v dy[v][co] * x[v + tap][ci].
//
// GEMM view (the reduction runs over VOXELS, so both operands are MN-major):
//   D[(kd,ci)][co] (+)= A[(kd,ci)][16 voxels] * B[16 voxels][co]          one tcgen05.mma per (kh,kw) tap
//   * the C8-planar activation layout ([..][C/8][H][W][8] bf16) is exactly the canonical no-swizzle
//     MN-major UMMA core matrix: 8 consecutive voxels of a W row x 8 channels = 128 contiguous bytes.
//     One K step = two such row segments one tile row apart (LBO = row pitch); channel groups (and the
//     kd depth planes, landed back to back by ONE 5-D TMA box with zero fill outside the volume) are the
//     M groups at a uniform stride (SBO = halo'd plane bytes).
//   * the 9 in-plane taps are the SAME shared-memory tile read through descriptors whose start address is
//     shifted by (kh*pitch + kw*16) bytes; each tap owns its own TMEM accumulator (9*N columns).
//   * a CTA keeps its accumulators in TMEM across ALL the voxel tiles of its split-K slice and touches
//     global memory once at the end (fp32 atomics into dW).
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer (+TMEM alloc), warps 2..5 epilogue.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kThreadsW = 192;
constexpr int kMaxStagesW = 8;
constexpr int kSmemBudgetW = 220 * 1024;

struct WgCfg {
    int th, tw;            // tile rows (even) / cols (multiple of 8)
    int nkd;               // depth taps per M tile (kd or 1)
    int c8chunk;           // channel groups per M tile and depth tap
    int mtiles_c, mtiles_kd;
    int m;                 // UMMA M (64 or 128)
    int nb, nchunks;       // UMMA N, number of N chunks
    int plane_x, plane_dy; // bytes of one channel-group plane in the x / dy tile
    int dy_off;            // offset of the dy tile inside a stage (x bytes rounded up to 128)
    int x_bytes, dy_bytes, stage_bytes, stages, pad_bytes, smem_bytes;
    int tmem_cols;
    int ndy;               // depth-stacked mode: ndy dy planes x (ndy + kd - 1) x planes per tile (see the kernel); 1 = off
    int ncols;             // UMMA N = nb * ndy
};

bool make_wg_cfg(int h, int w, int cin, int cout, int kd, int allow_pair, WgCfg& c) {
    if (cin % 8 != 0 || (cout % 16 != 0 && cout != 8) || cin <= 0 || cout <= 0) return false;
    c.tw = w >= 32 ? 32 : (w >= 16 ? 16 : 8);
    c.th = h >= 8 ? 8 : ((h + 1) / 2) * 2;
    const int g_all = cin / 8;
    // depth stacking: k3 -> 2 dy planes x 4 x planes (3 of the 4 blocks per dy plane are taps); k(1,3,3) -> the diagonal
    // blocks of ndy x ndy planes (4 planes when the output is one channel group: the head's classes padded to 8)
    c.ndy = 1;
    if (allow_pair && kd == 3 && g_all <= 4 && cout % 16 == 0) c.ndy = 2;
    else if (allow_pair && kd == 1 && cout == 8 && g_all <= 2) c.ndy = 4;
    else if (allow_pair && kd == 1 && cout == 8 && g_all <= 4) c.ndy = 2;
    else if (allow_pair && kd == 1 && cout == 16 && g_all <= 8) c.ndy = 2;
    if (c.ndy > 1) { c.nkd = c.ndy + kd - 1; c.c8chunk = g_all; c.mtiles_kd = 1; c.mtiles_c = 1; }
    else if (kd * g_all <= 16) { c.nkd = kd; c.c8chunk = g_all; c.mtiles_kd = 1; c.mtiles_c = 1; }
    else {
        c.nkd = 1; c.mtiles_kd = kd;
        c.c8chunk = g_all < 16 ? g_all : 16;
        if (g_all % c.c8chunk != 0) return false;
        c.mtiles_c = g_all / c.c8chunk;
    }
    const int groups = c.nkd * c.c8chunk;
    c.m = groups <= 8 ? 64 : 128;
    if (cout == 8 && c.m != 64) return false;          // N = 8 needs the M = 64 shape
    c.nb = cout == 8 ? 8 : ((cout % 32 == 0 && c.ndy == 1) ? 32 : 16);
    c.ncols = c.ndy * c.nb;
    c.nchunks = cout / c.nb;
    if (groups > 8 && c.tw == 32 && cin >= 32 && h * w >= 128 * 128) c.tw = 16;   // keep >= 3 stages at full resolution
    c.plane_x = (c.th + 2) * (c.tw + 2) * 16;
    c.plane_dy = c.th * c.tw * 16;
    c.x_bytes = groups * c.plane_x;
    c.dy_bytes = (c.ncols / 8) * c.plane_dy;
    c.dy_off = ((c.x_bytes + 127) / 128) * 128;
    c.stage_bytes = ((c.dy_off + c.dy_bytes + 127) / 128) * 128;
    // the M=64/128 operand reads 8/16 channel-group planes from the tile start: keep that window inside the allocation
    int over = (c.m / 8 + 1) * c.plane_x - c.stage_bytes;
    c.pad_bytes = over > 0 ? ((over + 127) / 128) * 128 : 0;
    c.stages = (kSmemBudgetW - c.pad_bytes - 2048) / c.stage_bytes;
    if (c.stages > kMaxStagesW) c.stages = kMaxStagesW;
    if (c.stages < 2) return false;
    c.smem_bytes = c.stages * c.stage_bytes + c.pad_bytes + 1024 + 256;
    int cols = 9 * c.ncols;
    c.tmem_cols = 32;
    while (c.tmem_cols < cols) c.tmem_cols *= 2;
    return c.tmem_cols <= 512;
}

struct WgParams {
    float* dw;
    int N, D, H, W, cin, cout, kd;
    int x_c8off, dy_c8off;
    int th, tw, nkd, c8chunk, mtiles_c, mtiles_kd, m, nb, nchunks;
    int plane_x, plane_dy, x_bytes, dy_off, stage_bytes, stages, tmem_cols;
    int tiles_h, tiles_w, tiles_total, split;
    int ndy, ncols, dplanes;       // dplanes: tile index range along depth, ceil(D / ndy)
    int taps;                      // 9, or 1 = only the centre in-plane tap (k = (kd,1,1))
    int tapmajor;                  // dW written as [tap][cout][cin] (coalesced atomics; see fpl_wgrad_tapmajor_to_dw_batch)
};

struct WgWork {
    int mt_kd, mt_c, nc, slice;
};

__device__ __forceinline__ WgWork decode_work(const WgParams& P, int b) {
    WgWork w;
    w.slice = b % P.split; b /= P.split;
    w.nc = b % P.nchunks; b /= P.nchunks;
    w.mt_c = b % P.mtiles_c;
    w.mt_kd = b / P.mtiles_c;
    return w;
}

__global__ void __launch_bounds__(kThreadsW) conv3d_wgrad_tc_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                   const __grid_constant__ CUtensorMap dymap, WgParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    // barriers live in front of the stage ring so that operand over-reads past the last stage stay in the pad
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kMaxStagesW;
    uint64_t* done_bar = bars + 2 * kMaxStagesW;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStagesW + 1);
    uint8_t* ring = smem + 256;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const WgWork wk = decode_work(P, blockIdx.x);
    const int tile_begin = (int)(((int64_t)P.tiles_total * wk.slice) / P.split);
    const int tile_end = (int)(((int64_t)P.tiles_total * (wk.slice + 1)) / P.split);
    const int pad_d = P.kd / 2;
    const int kd0 = P.mtiles_kd > 1 ? wk.mt_kd : 0;          // first depth tap of this M tile

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&xmap) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&dymap) : "memory");
        for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(done_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    FPL_PDL_WAIT();      // prologue above overlapped the previous kernel's tail; from here on its results are visible
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int t = tile_begin; t < tile_end; ++t) {
                // depth runs fastest: consecutive tiles of a CTA are the same (h, w) window in consecutive depth steps, so
                // the x planes two neighbouring steps share (kd halo; 2 of 4 planes in the depth-stacked mode) are
                // re-fetched by the SAME SM right after their first use and hit L2 (w-fastest order: 293 MB of DRAM
                // reads for the 201 MB of up4.conv1, profiles/r02a_prof_wgrad_summary.md)
                int r = t;
                const int dp = r % P.dplanes; r /= P.dplanes;
                const int tw_i = r % P.tiles_w; r /= P.tiles_w;
                const int th_i = r % P.tiles_h;
                const int n = r / P.tiles_h;
                // stacked mode: dy planes ndy*dp .. ndy*dp+ndy-1 against x planes ndy*dp-pad .. (planes outside the
                // volume: TMA zero fill)
                const int d = P.ndy * dp;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* x_dst = ring + (size_t)stage * P.stage_bytes;
                uint8_t* dy_dst = x_dst + P.dy_off;
                mbar_expect_tx(&full_bar[stage], (uint32_t)(P.x_bytes + (P.ncols / 8) * P.plane_dy));
                tma_load_5d(x_dst, &xmap, &full_bar[stage], 2 * (tw_i * P.tw - 1), th_i * P.th - 1,
                            P.x_c8off + wk.mt_c * P.c8chunk, d + kd0 - pad_d, n);
                tma_load_5d(dy_dst, &dymap, &full_bar[stage], 2 * (tw_i * P.tw), th_i * P.th,
                            P.dy_c8off + wk.nc * (P.nb / 8), d, n);
                if (++stage == P.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: the whole warp runs the loop (uniform), one lane issues =====================
        // kind::f16, bf16 x bf16 -> fp32, A and B both MN-major (bits 15, 16)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                               ((uint32_t)(P.ncols >> 3) << 17) | ((uint32_t)(P.m >> 4) << 24);
        const uint32_t pitch_x = (uint32_t)(P.tw + 2) * 16, pitch_dy = (uint32_t)P.tw * 16;
        // descriptors = constant high part + (smem byte address >> 4) in the low 14 bits
        const uint64_t a_hi = make_desc(0, pitch_x, (uint32_t)P.plane_x), b_hi = make_desc(0, pitch_dy, (uint32_t)P.plane_dy);
        uint32_t tap_off[9];                                  // (kh*pitch + kw*16) >> 4
#pragma unroll
        for (int t9 = 0; t9 < 9; ++t9) tap_off[t9] = ((uint32_t)(t9 / 3) * pitch_x + (uint32_t)(t9 % 3) * 16) >> 4;
        uint32_t d_tap[9];
#pragma unroll
        for (int t9 = 0; t9 < 9; ++t9) d_tap[t9] = tmem_base + (uint32_t)(t9 * P.ncols);
        const uint32_t ring_u = smem_u32(ring);
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        uint32_t accumulate = 0;
        for (int t = tile_begin; t < tile_end; ++t) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t x_base = (ring_u + (uint32_t)stage * (uint32_t)P.stage_bytes) >> 4;
            const uint32_t dy_base = x_base + ((uint32_t)P.dy_off >> 4);
            for (int hp = 0; hp < P.th / 2; ++hp) {
                const uint32_t a_row = x_base + (((uint32_t)(2 * hp) * pitch_x) >> 4);
                const uint32_t b_row = dy_base + (((uint32_t)(2 * hp) * pitch_dy) >> 4);
                // 64-bit adds of warp-uniform values (the 14-bit start-address field never carries): uniform datapath
                uint64_t bdesc = b_hi + (uint64_t)b_row, a_col = a_hi + (uint64_t)a_row;
                for (int j = 0; j < P.tw / 8; ++j, bdesc += 8, a_col += 8) {
                    if (P.taps == 1) {
                        if (leader) umma_bf16(tmem_base, a_col + (uint64_t)tap_off[4], bdesc, idesc, accumulate);
                    } else {
#pragma unroll
                        for (int t9 = 0; t9 < 9; ++t9)
                            if (leader) umma_bf16(d_tap[t9], a_col + (uint64_t)tap_off[t9], bdesc, idesc, accumulate);
                    }
                    accumulate = 1;
                }
            }
            if (leader) umma_commit(&empty_bar[stage]);
            __syncwarp();
            if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
        if (leader) umma_commit(done_bar);
        __syncwarp();
        FPL_PDL_TRIGGER();   // this CTA has issued its last tile: the next kernel of the stream may be scheduled as SMs drain
    } else if (tile_end > tile_begin) {
        // ===================== epilogue: TMEM -> fp32 atomics into dW =====================
        const int quarter = warp & 3;
        mbar_wait(done_bar, 0);
        tc_fence_after();
        const int T = P.kd * P.taps;
        const int tlane = quarter * 32 + lane;               // TMEM lane this thread reads
        int row;                                             // M row held by that lane
        if (P.m == 128) row = tlane;
        else row = (lane < 16) ? quarter * 16 + lane : -1;   // M=64: 16 rows per 32-lane quadrant
        bool valid = row >= 0 && row < P.m;
        int kdi = 0, ci = 0;
        if (valid) {
            const int g = row >> 3;
            valid = g < P.nkd * P.c8chunk;
            kdi = kd0 + g / P.c8chunk;                       // pair mode: index of the x plane (0..3) inside the tile
            ci = (wk.mt_c * P.c8chunk + g % P.c8chunk) * 8 + (row & 7);
        }
        for (int t9 = 0; t9 < P.taps; ++t9) {
            for (int c0 = 0; c0 < P.ncols; c0 += 16) {
                uint32_t r[16];
                tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t9 * P.ncols + c0), r);
                tmem_ld_wait();
                // stacked mode: column block dd = col / nb is dy plane ndy*dp+dd, row block kdi is x plane ndy*dp-pad+kdi:
                // depth tap kd = kdi - dd (the (kdi, dd) blocks of one tap are summed by the atomics).  nb is a multiple
                // of 8, so each half of the 16 loaded columns lies in one block.
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int col = c0 + 8 * half;
                    const int dd = P.ndy > 1 ? col / P.nb : 0;
                    const int kd_tap = P.ndy > 1 ? kdi - dd : kdi;
                    const int co0 = wk.nc * P.nb + (col - dd * P.nb);
                    if (!(valid && kd_tap >= 0 && kd_tap < P.kd)) continue;
                    if (P.tapmajor) {
                        // lanes = consecutive input channels: one 128-byte line per warp instruction
                        float* base = P.dw + ((int64_t)(kd_tap * P.taps + t9) * P.cout + co0) * P.cin + ci;
#pragma unroll
                        for (int i = 0; i < 8; ++i) atomicAdd(base + (int64_t)i * P.cin, __uint_as_float(r[8 * half + i]));
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            atomicAdd(P.dw + ((int64_t)(co0 + i) * P.cin + ci) * T + kd_tap * P.taps + t9,
                                      __uint_as_float(r[8 * half + i]));
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
    }
}

CUresult encode_5d(EncodeTiledFn encode, CUtensorMap* map, const void* base, int n, int d, int c8tot, int h, int w,
                   int box_w, int box_h, int box_c8, int box_d) {
    // 8-byte elements (4 bf16 channels) so that a 34-voxel halo row fits the 256-element box limit
    cuuint64_t gdim[5] = {(cuuint64_t)w * 2, (cuuint64_t)h, (cuuint64_t)c8tot, (cuuint64_t)d, (cuuint64_t)n};
    cuuint64_t gstr[4] = {(cuuint64_t)w * 16, (cuuint64_t)h * w * 16, (cuuint64_t)c8tot * h * w * 16,
                          (cuuint64_t)d * c8tot * h * w * 16};
    cuuint32_t box[5] = {(cuuint32_t)box_w * 2, (cuuint32_t)box_h, (cuuint32_t)box_c8, (cuuint32_t)box_d, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

}  // namespace

bool fpl_wgrad_hs_eligible(int d, int h, int w, int cin, int cout, int kd, int taps);
int fpl_wgrad_hs_launch(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off, float* dw, int n,
                        int d, int h, int w, int cin, int cout, void* stream, int tapmajor);
bool fpl_wgrad_rs_eligible(int d, int h, int w, int cin, int cout, int kd, int taps);
int fpl_wgrad_rs_launch(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off, float* dw, int n,
                        int d, int h, int w, void* stream, int tapmajor);

static int wgrad_tc_launch(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                           float* dw, int n, int d, int h, int w, int cin, int cout, int kd, int taps, void* stream,
                           int tapmajor = 0) {
    FPL_REQUIRE(kd == 1 || kd == 3, "fpl_conv3d_wgrad_tc: kd=%d must be 1 or 3", kd);
    if (fpl_wgrad_hs_eligible(d, h, w, cin, cout, kd, taps))
        return fpl_wgrad_hs_launch(x, x_c8tot, x_c8off, dy, dy_c8tot, dy_c8off, dw, n, d, h, w, cin, cout, stream, tapmajor);
    if (fpl_wgrad_rs_eligible(d, h, w, cin, cout, kd, taps))
        return fpl_wgrad_rs_launch(x, x_c8tot, x_c8off, dy, dy_c8tot, dy_c8off, dw, n, d, h, w, stream, tapmajor);
    WgCfg c;
    FPL_REQUIRE(make_wg_cfg(h, w, cin, cout, kd, d >= 2, c),
                "fpl_conv3d_wgrad_tc: unsupported shape (cin %d, cout %d, %dx%d)", cin, cout, h, w);
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0,
                "fpl_conv3d_wgrad_tc: x/dy must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_conv3d_wgrad_tc: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap xmap, dymap;
    CUresult r = encode_5d(encode, &xmap, x, n, d, x_c8tot, h, w, c.tw + 2, c.th + 2, c.c8chunk, c.nkd);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_wgrad_tc: tensor map (x) failed (%d)", (int)r);
    r = encode_5d(encode, &dymap, dy, n, d, dy_c8tot, h, w, c.tw, c.th, c.nb / 8, c.ndy);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_wgrad_tc: tensor map (dy) failed (%d)", (int)r);
    WgParams P;
    P.dw = dw;
    P.N = n; P.D = d; P.H = h; P.W = w; P.cin = cin; P.cout = cout; P.kd = kd;
    P.x_c8off = x_c8off; P.dy_c8off = dy_c8off;
    P.th = c.th; P.tw = c.tw; P.nkd = c.nkd; P.c8chunk = c.c8chunk; P.mtiles_c = c.mtiles_c; P.mtiles_kd = c.mtiles_kd;
    P.m = c.m; P.nb = c.nb; P.nchunks = c.nchunks; P.plane_x = c.plane_x; P.plane_dy = c.plane_dy; P.x_bytes = c.x_bytes; P.dy_off = c.dy_off;
    P.stage_bytes = c.stage_bytes; P.stages = c.stages; P.tmem_cols = c.tmem_cols;
    P.tiles_h = (h + c.th - 1) / c.th; P.tiles_w = (w + c.tw - 1) / c.tw;
    P.ndy = c.ndy; P.ncols = c.ncols; P.dplanes = (d + c.ndy - 1) / c.ndy;
    int64_t tiles = (int64_t)P.tiles_h * P.tiles_w * P.dplanes * n;
    FPL_REQUIRE(tiles < (1ll << 30), "fpl_conv3d_wgrad_tc: too many tiles");
    P.tiles_total = (int)tiles;
    const int pairs = c.mtiles_kd * c.mtiles_c * c.nchunks;
    // split-K over voxel tiles: every CTA ends with 9*128*N atomics into dW, so a slice should own >= 2 tiles (measured
    // with a tuning tool that has since been removed)
    // (deep levels: few tiles, many (M,N) pairs -> split 1; full resolution: one CTA per SM)
    int split = FPL_NUM_SMS / pairs;
    if (split > P.tiles_total / 2) split = P.tiles_total / 2;
    if (split < 1) split = 1;
    P.split = split;
    P.taps = taps; P.tapmajor = tapmajor;
    FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, c.smem_bytes));
    fpl_launch(conv3d_wgrad_tc_kernel, pairs * split, kThreadsW, c.smem_bytes, (cudaStream_t)stream, xmap, dymap, P);
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_conv3d_wgrad_tc(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                                   float* dw, int n, int d, int h, int w, int cin, int cout, int kd, void* stream) {
    return wgrad_tc_launch(x, x_c8tot, x_c8off, dy, dy_c8tot, dy_c8off, dw, n, d, h, w, cin, cout, kd, 9, stream);
}

/* wgrad of a k = (3,1,1) conv: dW[cout][cin][3] (fp32, ACCUMULATED into); one MMA per K step instead of nine. */
extern "C" int fpl_conv3d_wgrad_tc_k311(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                                        float* dw, int n, int d, int h, int w, int cin, int cout, void* stream) {
    return wgrad_tc_launch(x, x_c8tot, x_c8off, dy, dy_c8tot, dy_c8off, dw, n, d, h, w, cin, cout, 3, 1, stream);
}

/* fpl_conv3d_wgrad_tc writing a TAP-MAJOR scratch gradient  S[kd*9 + t9][cout][cin]  (fp32, ACCUMULATED into): the
 * epilogue's atomics then hit consecutive addresses across a warp (input channels are the TMEM lanes).  The scratch
 * of all layers is folded into the PyTorch layout by ONE fpl_wgrad_tapmajor_to_dw_batch launch. */
extern "C" int fpl_conv3d_wgrad_tc_tapmajor(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                                            float* scratch, int n, int d, int h, int w, int cin, int cout, int kd,
                                            void* stream) {
    return wgrad_tc_launch(x, x_c8tot, x_c8off, dy, dy_c8tot, dy_c8off, scratch, n, d, h, w, cin, cout, kd, 9, stream, 1);
}

namespace {
constexpr int kMaxFold = 64;
struct FoldBatch {
    const float* s[kMaxFold];
    float* dw[kMaxFold];
    int cout[kMaxFold], cin[kMaxFold], taps[kMaxFold], scout[kMaxFold];
};
// dW[row][tap] += S[tap][row]   (blockIdx.y = layer; row = co*cin + ci; S has scout >= cout rows of cin per tap, the first
// cout are folded).  Both sides are coalesced through a shared-memory transpose: a block owns kFoldRows consecutive
// rows, reads them tap by tap (consecutive threads = consecutive rows) and writes the [rows][taps] block contiguously.
// Negative tap count: nn.ConvTranspose3d layout, row = ci*cout + co (small tensors; the gather is left uncoalesced).
constexpr int kFoldRows = 256;
__global__ void __launch_bounds__(256) fold_tapmajor_kernel(const __grid_constant__ FoldBatch B) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    __shared__ float tile[kFoldRows * 27];
    const int e = blockIdx.y;
    const float* __restrict__ s = B.s[e];
    float* dw = B.dw[e];
    const int cout = B.cout[e], cin = B.cin[e];
    const bool transposed = B.taps[e] < 0;
    const int T = transposed ? -B.taps[e] : B.taps[e];
    const int Tp = T | 1;                                   // odd row pitch: conflict-free transposed writes
    const uint32_t magic = 0xffffffffu / (uint32_t)T + 1u;  // i / T == umulhi(i, magic) for i < 2^16
    const int rows = cout * cin;
    const int64_t tap_stride = (int64_t)B.scout[e] * cin;
    for (int r0 = blockIdx.x * kFoldRows; r0 < rows; r0 += gridDim.x * kFoldRows) {
        const int nr = min(kFoldRows, rows - r0);
        const int r = threadIdx.x;
        if (r < nr) {
            int src = r0 + r;
            if (transposed) {
                const int ci = src / cout, co = src - ci * cout;
                src = co * cin + ci;
            }
            const float* sp = s + src;
            if (T == 27) {                                  // all 27 loads of a row in flight
                float t27[27];
#pragma unroll
                for (int tap = 0; tap < 27; ++tap) t27[tap] = __ldg(sp + tap * tap_stride);
#pragma unroll
                for (int tap = 0; tap < 27; ++tap) tile[r * Tp + tap] = t27[tap];
            } else {
#pragma unroll 9
                for (int tap = 0; tap < T; ++tap) tile[r * Tp + tap] = __ldg(sp + tap * tap_stride);
            }
        }
        __syncthreads();
        float* out = dw + (int64_t)r0 * T;
        // read-modify-write in batches of 9 independent loads per thread (one load -> add -> store per iteration is a
        // memory round trip each: 27 of them in a row paced the kernel at 1.5 TB/s)
        const int total = nr * T;
        for (int i0 = threadIdx.x; i0 < total; i0 += 9 * (int)blockDim.x) {
            float v[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                const int i = i0 + k * (int)blockDim.x;
                v[k] = i < total ? out[i] : 0.0f;
            }
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                const int i = i0 + k * (int)blockDim.x;
                if (i < total) {
                    const int rr = (int)__umulhi((uint32_t)i, magic), tap = i - rr * T;
                    out[i] = v[k] + tile[rr * Tp + tap];
                }
            }
        }
        __syncthreads();
    }
}
}  // namespace

extern "C" int fpl_wgrad_tapmajor_to_dw_batch(int count, const float* const* h_scratch, float* const* h_dw, const int* h_cout,
                                              const int* h_cin, const int* h_taps, const int* h_scratch_cout, void* stream) {
    FPL_REQUIRE(count >= 0 && count <= kMaxFold, "fpl_wgrad_tapmajor_to_dw_batch: count %d not in [0,%d]", count, kMaxFold);
    if (count == 0) return 0;
    FoldBatch B;
    int max_total = 0;
    for (int e = 0; e < count; ++e) {
        B.s[e] = h_scratch[e]; B.dw[e] = h_dw[e]; B.cout[e] = h_cout[e]; B.cin[e] = h_cin[e]; B.taps[e] = h_taps[e];
        B.scout[e] = h_scratch_cout != nullptr ? h_scratch_cout[e] : h_cout[e];
        FPL_REQUIRE((h_taps[e] < 0 ? -h_taps[e] : h_taps[e]) <= 27 && h_taps[e] != 0, "fpl_wgrad_tapmajor_to_dw_batch: tap count %d out of range", h_taps[e]);
        FPL_REQUIRE(B.scout[e] >= B.cout[e], "fpl_wgrad_tapmajor_to_dw_batch: scratch rows %d < folded rows %d", B.scout[e], B.cout[e]);
        const int total = h_cout[e] * h_cin[e] * (h_taps[e] < 0 ? -h_taps[e] : h_taps[e]);
        if (total > max_total) max_total = total;
    }
    int bx = (max_total / 9 + kFoldRows - 1) / kFoldRows;      // ~ blocks of kFoldRows rows for the largest layer
    if (bx > 296) bx = 296;
    if (bx < 1) bx = 1;
    fpl_launch(fold_tapmajor_kernel, dim3(bx, count), 256, 0, (cudaStream_t)stream, B);
    FPL_LAUNCH_CHECK();
    return 0;
}

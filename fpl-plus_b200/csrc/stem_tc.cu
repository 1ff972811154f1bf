// Tensor-core forward and weight gradient of the network's FIRST conv, nn.Conv3d(1 -> 16, k3, p1) on the fp32 NCDHW image
// (PyMIC/pymic/net/net3d/unet2d5_dsbn.py:75 with in_chns = 1, and its autograd), WITHOUT a materialised patch tensor.
//
// A 1-channel input has no channel dimension to reduce over, so the GEMM's K is the 27 taps: builder warps gather, per
// voxel, the 27 neighbours of the image from a rolling window of staged halo planes (every image value split ONCE into a
// bf16 value + bf16 residual word) and write them as four 16-byte vectors of 8 taps (value) + four more (residual):
// [hi g0..g3 | lo g0..g3][16 rows][32 voxels][8 taps].  That ONE layout is
//   * the K-major A operand of the forward:  y[v][co] = sum_k A[v][k] W[k][co]   (M = 128 voxels = 4 rows, six K steps:
//     hi x w_hi, lo x w_hi, hi x w_lo: fp32-accurate although every operand is bf16), and
//   * the MN-major A operand of the weight gradient:  dW[k][co] = sum_v A[v][k] dy[v][co]   (M = 64 = hi | lo taps,
//     K = 16 voxels of a row, B = the dy tile straight from TMA), hi and lo rows summed by the final atomics.
// Before: fpl_patch9_c8 wrote a 64 B/voxel patch tensor (24 us), a k(3,1,1) tensor-core conv read it (50 us) and so did
// the k(3,1,1) wgrad (40 us): 343 + 201 MB of traffic per pass for 75 + 75 MB of algorithmic bytes.
// A CTA walks CONSECUTIVE tiles, depth fastest: tile coordinates are stepped, not divided, and a tile that continues its
// column loads one new image plane instead of three.  41 us forward / 35 us weight gradient at 4x32x128x128 (first version:
// 66 / 50 us with a per-tap split, generic shared-memory addressing, three divisions per tile and role, a spilling epilogue;
// ncu: 640 instructions per voxel-warp, 60 % issue slots busy -- profiles/README.md round 2e).
// Warp roles: forward: warp 0 MMA issuer, warps 1..8 epilogue (+bias, bf16 store, BatchNorm sums), warps 9..24 builders;
//             wgrad:   warp 0 MMA issuer, warp 1 TMA producer (dy), warps 2..5 final epilogue, warps 6..21 builders.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kSR = 16, kSC = 32;                       // tile: 16 rows x 32 voxels of one plane
constexpr int kSGroup = kSR * kSC * 16;                 // one 8-tap group plane of the tile: 8192 bytes
constexpr int kSStage = 8 * kSGroup;                    // hi g0..3 | lo g0..3
constexpr int kSHaloR = kSR + 2, kSHaloC = kSC + 2, kSHalo = 3 * kSHaloR * kSHaloC;     // staged image tile (floats)
constexpr int kSBuild = 16;                             // builder warps: one voxel of the tile per builder thread

struct StemTile {
    int n, z, h0, w0;
};

struct StemGeo {
    int N, D, H, W, tiles_h, tiles_w, total_tiles;
};

__device__ __forceinline__ StemTile stem_tile(const StemGeo& G, int t) {
    StemTile c;
    c.z = t % G.D; t /= G.D;                            // depth fastest: consecutive tiles of a CTA share two image planes (L1 / L2)
    const int tw = t % G.tiles_w; t /= G.tiles_w;
    const int th = t % G.tiles_h;
    c.n = t / G.tiles_h;
    c.h0 = th * kSR; c.w0 = tw * kSC;
    return c;
}

// the next tile in depth-fastest order (the tiles a CTA walks are consecutive: no divisions in the loops)
__device__ __forceinline__ void stem_tile_next(const StemGeo& G, StemTile& c) {
    if (++c.z == G.D) {
        c.z = 0;
        c.w0 += kSC;
        if (c.w0 >= G.tiles_w * kSC) {
            c.w0 = 0;
            c.h0 += kSR;
            if (c.h0 >= G.tiles_h * kSR) { c.h0 = 0; ++c.n; }
        }
    }
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// The builders keep a ROLLING window of image planes in shared memory: a ring of four (18 x 34) halo planes, plane z in
// slot (z + 1) & 3.  The tiles a CTA walks are consecutive in depth, so a tile that continues its column needs ONE new plane
// (z + 1); the first tile of a column (or of the CTA) loads all three.  Builder thread b owns the plane elements b and
// b + 512 (< 612): their (row, column) is the same for every plane and tile: decoded ONCE into a packed word
// (row + 1) | (column + 1) << 8 (negative = beyond the plane) and the element offset from the tile origin.
constexpr int kSPlane = kSHaloR * kSHaloC;                                                // 612 values
constexpr int kSLoadsP = (kSPlane + 32 * kSBuild - 1) / (32 * kSBuild);                   // 2 per thread and plane
static_assert(4 * kSPlane <= 2 * kSHalo, "the plane ring fits the staged-tile allocation");

struct StemHaloIdx {
    int code[kSLoadsP], off[kSLoadsP];
};

__device__ __forceinline__ void stem_halo_idx(int b, const StemGeo& G, StemHaloIdx& I) {
#pragma unroll
    for (int u = 0; u < kSLoadsP; ++u) {
        const int i = b + u * 32 * kSBuild;
        const int cw = i % kSHaloC - 1, rh = i / kSHaloC - 1;
        I.code[u] = i < kSPlane ? (rh + 1) | ((cw + 1) << 8) : -1;
        I.off[u] = i < kSPlane ? rh * G.W + cw : 0;
    }
}

// image planes c.z - 1 .. c.z + 1 (full) or c.z + 1 only, into regs[plane][u]
__device__ __forceinline__ void stem_load_planes(const float* __restrict__ img, const StemGeo& G, const StemTile& c, const StemHaloIdx& I,
                                                 bool full, float* regs) {
    const int64_t HW = (int64_t)G.H * G.W;
    const float* base = img + ((int64_t)c.n * G.D + c.z) * HW + (int64_t)c.h0 * G.W + c.w0;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        if (p < 2 && !full) continue;
        const bool zok = (unsigned)(c.z + p - 1) < (unsigned)G.D;
        const float* pb = base + (int64_t)(p - 1) * HW;
#pragma unroll
        for (int u = 0; u < kSLoadsP; ++u) {
            const int code = I.code[u];
            const int h = c.h0 + (code & 255) - 1, w = c.w0 + (code >> 8) - 1;
            float v = 0.0f;
            if (code >= 0 && zok && (unsigned)h < (unsigned)G.H && (unsigned)w < (unsigned)G.W) v = __ldg(pb + I.off[u]);
            regs[p * kSLoadsP + u] = v;
        }
    }
}

// The staged image tile holds one 32-bit word per image value: low half = bf16(value) (hi), high half = bf16(value - hi)
// (lo): hi + lo carries 16 mantissa bits -- the same split as fpl_patch9_c8, so the products the tensor pipe forms are
// those of the patch-tensor path.  Splitting once per image value (instead of once per tap: 27x) leaves the builders two
// byte permutes per tap pair.
__device__ __forceinline__ uint32_t stem_split(float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    return (uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(l) << 16);
}

__device__ __forceinline__ void stem_stage_planes(uint32_t halo_addr, int b, int z, bool full, const float* regs) {
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        if (p < 2 && !full) continue;
        const uint32_t slot = halo_addr + 4u * (uint32_t)(((z + p) & 3) * kSPlane);
#pragma unroll
        for (int u = 0; u < kSLoadsP; ++u) {
            const int i = b + u * 32 * kSBuild;
            if (i < kSPlane) sts_u32(slot + 4u * (uint32_t)i, stem_split(regs[p * kSLoadsP + u]));
        }
    }
}

// the 8 tap vectors (4 hi, 4 lo) of the voxel builder thread b owns: (row b / 32, col b % 32) of the tile at depth z;
// shared-state-space addresses (generic pointers into the dynamic array cost a descriptor move per access here)
__device__ __forceinline__ void stem_build(uint32_t halo_addr, uint32_t stage_addr, int b, int z) {
    const int row = b >> 5, col = b & 31;
    uint32_t t[28];
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
        const uint32_t src = halo_addr + 4u * (uint32_t)(((z + kd) & 3) * kSPlane + row * kSHaloC + col);
#pragma unroll
        for (int k = 0; k < 9; ++k) t[kd * 9 + k] = lds_u32(src + 4u * (uint32_t)((k / 3) * kSHaloC + k % 3));
    }
    t[27] = 0u;
    uint32_t hi[16], lo[16];                                   // packed bf16 pairs, taps 2i and 2i+1
#pragma unroll
    for (int i = 0; i < 14; ++i) {
        hi[i] = __byte_perm(t[2 * i], t[2 * i + 1], 0x5410);
        lo[i] = __byte_perm(t[2 * i], t[2 * i + 1], 0x7632);
    }
    hi[14] = hi[15] = lo[14] = lo[15] = 0u;
    const uint32_t dst = stage_addr + 16u * (uint32_t)(row * kSC + col);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        sts_v4(dst + (uint32_t)(g * kSGroup), hi[4 * g], hi[4 * g + 1], hi[4 * g + 2], hi[4 * g + 3]);
        sts_v4(dst + (uint32_t)((4 + g) * kSGroup), lo[4 * g], lo[4 * g + 1], lo[4 * g + 2], lo[4 * g + 3]);
    }
}

// one builder iteration protocol shared by the forward and the weight gradient (see the kernels): returns nothing; the
// caller owns the stage ring and its barriers
#define STEM_BUILDER_LOOP(STAGE_ADDR, FULL_BAR, N_STAGES)                                                              \
    float regs[3 * kSLoadsP];                                                                                          \
    StemHaloIdx I;                                                                                                     \
    stem_halo_idx(b, G, I);                                                                                            \
    const uint32_t halo_u = smem_u32(halo), ring_a = smem_u32(ring);                                                   \
    int stage = 0; uint32_t phase = 0;                                                                                 \
    StemTile c = stem_tile(G, tile_begin);                                                                             \
    bool full = true;                                                                                                  \
    if (tile_begin < tile_end) stem_load_planes(P.img, G, c, I, true, regs);                                           \
    for (int t = tile_begin; t < tile_end; ++t) {                                                                      \
        /* a new column overwrites ring slots the previous column's last tile may still be read from */               \
        if (full && t != tile_begin) asm volatile("bar.sync 2, %0;" ::"n"(32 * kSBuild) : "memory");                   \
        stem_stage_planes(halo_u, b, c.z, full, regs);                                                                 \
        /* the next tile's image floats travel while this tile is built */                                            \
        StemTile nx = c;                                                                                               \
        stem_tile_next(G, nx);                                                                                         \
        const bool nfull = nx.z == 0;                                                                                  \
        if (t + 1 < tile_end) stem_load_planes(P.img, G, nx, I, nfull, regs);                                          \
        asm volatile("bar.sync 2, %0;" ::"n"(32 * kSBuild) : "memory");                                                \
        mbar_wait(&empty_bar[stage], phase ^ 1);                                                                       \
        stem_build(halo_u, ring_a + (uint32_t)(STAGE_ADDR), b, c.z);                                                   \
        fence_proxy_async();                                                                                           \
        __syncwarp();                                                                                                  \
        if (lane == 0) mbar_arrive(&FULL_BAR[stage]);                                                                  \
        if (++stage == N_STAGES) { stage = 0; phase ^= 1; }                                                            \
        c = nx;                                                                                                        \
        full = nfull;                                                                                                  \
    }

// ------------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------------
constexpr int kSfThreads = 32 * (1 + 8 + kSBuild);
constexpr int kSfStages = 2;                            // 2 x 64 KB operand stages; 800 threads need up to 80 registers, so one CTA per SM

struct StemFwdParams {
    const float* img;          // [N][1][D][H][W]
    const float* w;            // [16][1][3][3][3]
    const float* bias;         // [16] or NULL
    bf16x8* y;                 // C8-planar slice (y_c8tot, y_c8off), 16 channels
    double* stats;             // [2][16] sum / sum of squares, ACCUMULATED (may be NULL)
    int y_c8tot, y_c8off;
    StemGeo G;
};

__global__ void __launch_bounds__(kSfThreads) stem_fwd_tc_kernel(StemFwdParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* ring = smem;                                                    // [stage][8 groups][16][32][16 B]
    uint8_t* b_sm = ring + kSfStages * kSStage;                              // [6 K steps][2 groups][16 co][8 taps] bf16
    float* halo = reinterpret_cast<float*>(b_sm + 6 * 512);                  // ring of 4 halo planes [18][34], split words (stem_split)
    uint64_t* bars = reinterpret_cast<uint64_t*>(halo + 2 * kSHalo);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kSfStages;
    uint64_t* tmem_full = bars + 2 * kSfStages;
    uint64_t* tmem_empty = bars + 2 * kSfStages + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kSfStages + 4);
    float* bias_sm = reinterpret_cast<float*>(bars + 2 * kSfStages + 6);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kSfStages; ++s) { mbar_init(&full_bar[s], kSBuild); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 8); }
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 128u);                              // 2 sets x 4 M tiles x 16 columns
    FPL_PDL_WAIT();
    {   // B: K step s = A groups {hi01, hi23, lo01, lo23, hi01, hi23} x weights {w_hi, w_hi, w_hi, w_hi, w_lo, w_lo} of tap groups {01, 23, ...}
        __nv_bfloat16* b = reinterpret_cast<__nv_bfloat16*>(b_sm);
        for (int i = threadIdx.x; i < 6 * 2 * 16 * 8; i += kSfThreads) {
            int t = i;
            const int j = t & 7; t >>= 3;
            const int co = t & 15; t >>= 4;
            const int gg = t & 1, s = t >> 1;
            const int k = ((s & 1) * 2 + gg) * 8 + j;
            const float v = k < 27 ? P.w[co * 27 + k] : 0.0f;
            const __nv_bfloat16 hi = __float2bfloat16_rn(v);
            b[i] = s < 4 ? hi : __float2bfloat16_rn(v - __bfloat162float(hi));
        }
        if (threadIdx.x < 16) bias_sm[threadIdx.x] = P.bias != nullptr ? P.bias[threadIdx.x] : 0.0f;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const StemGeo G = P.G;
    const int64_t HW = (int64_t)G.H * G.W;
    // consecutive tiles per CTA (depth fastest): the loops step the tile coordinates instead of dividing, and a CTA's
    // next tile shares two of its three image planes with the current one (L1)
    const int tile_begin = (int)(((int64_t)G.total_tiles * blockIdx.x) / gridDim.x);
    const int tile_end = (int)(((int64_t)G.total_tiles * (blockIdx.x + 1)) / gridDim.x);

    if (warp == 0) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(16 >> 3) << 17) | (8u << 24);
        const uint64_t a_hi = make_desc(0, kSGroup, 128), b_hi = make_desc(0, 256, 128);
        const uint64_t b0 = b_hi + (uint64_t)(smem_u32(b_sm) >> 4);
        const uint32_t ring_u = smem_u32(ring) >> 4;
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = tile_begin; t < tile_end; ++t) {
            mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t a0 = a_hi + (uint64_t)(ring_u + (uint32_t)((stage * kSStage) >> 4));
#pragma unroll
            for (int m = 0; m < 4; ++m) {
#pragma unroll
                for (int s = 0; s < 6; ++s) {
                    const int ga = s == 0 || s == 4 ? 0 : (s == 1 || s == 5 ? 2 : (s == 2 ? 4 : 6));
                    const uint64_t ad = a0 + (uint64_t)(ga * (kSGroup / 16) + m * (4 * kSC * 16 / 16));
                    if (leader) umma_bf16(tmem_base + (uint32_t)(acc * 64 + m * 16), ad, b0 + (uint64_t)(s * 32), idesc, s ? 1u : 0u);
                }
            }
            if (leader) { umma_commit(&empty_bar[stage]); umma_commit(&tmem_full[acc]); }
            __syncwarp();
            if (++stage == kSfStages) { stage = 0; phase ^= 1; }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        FPL_PDL_TRIGGER();
    } else if (warp <= 8) {
        // ===================== epilogue: + bias, bf16 C8-planar store, BatchNorm sums =====================
        // two warps per TMEM lane quadrant, one per channel group (8 of the 16 accumulator columns): 16 statistics
        // accumulators + 8 values per thread keep the 800-thread CTA inside 80 registers without spills
        const int quarter = warp & 3, half = (warp - 1) >> 2;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 8);
        float tacc[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) tacc[i] = 0.0f;
        float bias_r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) bias_r[i] = bias_sm[half * 8 + i];
        int acc = 0; uint32_t acc_phase = 0;
        StemTile c = stem_tile(G, tile_begin);
        for (int t = tile_begin; t < tile_end; ++t, stem_tile_next(G, c)) {
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const int w = c.w0 + lane;
            bf16x8* out0 = P.y + (((int64_t)c.n * G.D + c.z) * P.y_c8tot + P.y_c8off + half) * HW + w;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int h = c.h0 + 4 * m + quarter;
                const bool valid = h < G.H && w < G.W;
                uint32_t r[8];
                tmem_ld8(lane_base + (uint32_t)(acc * 64 + m * 16), r);
                tmem_ld_wait();
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]) + bias_r[i];
                if (valid) {
                    st_bf16x8(out0 + (int64_t)h * G.W, v);
#pragma unroll
                    for (int i = 0; i < 8; ++i) { tacc[i] += v[i]; tacc[8 + i] = fmaf(v[i], v[i], tacc[8 + i]); }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (P.stats != nullptr) {
            // one double atomic per channel and CTA: the 8 epilogue warps are first summed in shared memory (1184 warps
            // adding to the same 32 addresses serialise in the L2 atomic unit)
#pragma unroll
            for (int i = 0; i < 16; ++i) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) tacc[i] += __shfl_xor_sync(0xffffffffu, tacc[i], o);
            }
            float mine = 0.0f;                                    // lane e < 16: entry e = [sum | sum of squares][8 channels]
#pragma unroll
            for (int i = 0; i < 16; ++i) mine = lane == i ? tacc[i] : mine;
            float* red = halo;                                    // the builders are done with the image tiles: see the barrier
            asm volatile("bar.sync 3, 256;" ::: "memory");        // (all epilogue warps past their last tile; builders finish
                                                                  //  before the last tmem_full, which the epilogue has consumed)
            if (lane < 16) red[(warp - 1) * 16 + lane] = mine;
            asm volatile("bar.sync 3, 256;" ::: "memory");
            if (warp == 1) {
                const int stat = lane >> 4, ch = lane & 15, e = stat * 8 + (ch & 7), w0 = (ch >> 3) * 4;
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < 4; ++k) s += (double)red[(w0 + k) * 16 + e];
                atomicAdd(P.stats + stat * 16 + ch, s);
            }
        }
    } else {
        // ===================== builders =====================
        const int b = threadIdx.x - 32 * 9;
        STEM_BUILDER_LOOP(stage * kSStage, full_bar, kSfStages)
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 128u);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// weight gradient
// ------------------------------------------------------------------------------------------------------------------
constexpr int kSwThreads = 32 * (2 + 4 + kSBuild);
constexpr int kSwStages = 2;
constexpr int kSwDy = 2 * kSGroup;                      // dy tile: 2 channel groups x 16 x 32 vectors

struct StemWgParams {
    const float* img;
    float* dw;                 // [16][1][3][3][3], ACCUMULATED into
    int dy_c8off;
    StemGeo G;
    int split;
};

__global__ void __launch_bounds__(kSwThreads) stem_wgrad_tc_kernel(const __grid_constant__ CUtensorMap dymap, StemWgParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* ring = smem;                                                    // [stage][A: 8 groups | dy: 2 groups]
    float* halo = reinterpret_cast<float*>(ring + kSwStages * (kSStage + kSwDy));
    uint64_t* bars = reinterpret_cast<uint64_t*>(halo + 2 * kSHalo);
    uint64_t* full_a = bars;                                                 // builders -> MMA
    uint64_t* full_b = bars + kSwStages;                                     // TMA -> MMA
    uint64_t* empty_bar = bars + 2 * kSwStages;                              // MMA -> builders and producer (count 1, commit)
    uint64_t* done_bar = bars + 3 * kSwStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kSwStages + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const StemGeo G = P.G;
    const int tile_begin = (int)(((int64_t)G.total_tiles * blockIdx.x) / P.split);
    const int tile_end = (int)(((int64_t)G.total_tiles * (blockIdx.x + 1)) / P.split);
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&dymap) : "memory");
        for (int s = 0; s < kSwStages; ++s) { mbar_init(&full_a[s], kSBuild); mbar_init(&full_b[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(done_bar, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 32u);
    FPL_PDL_WAIT();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== MMA issuer: D[64 = hi | lo taps][16 co] += A^T[16 voxels] * dy[16 voxels] =====================
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(16 >> 3) << 17) |
                               ((uint32_t)(64 >> 4) << 24);
        // MN-major: LBO = the two 8-voxel core matrices of a K step (contiguous), SBO = group plane
        const uint64_t hi = make_desc(0, 128u, kSGroup);
        const uint32_t ring_u = smem_u32(ring) >> 4;
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        uint32_t accumulate = 0;
        for (int t = tile_begin; t < tile_end; ++t) {
            mbar_wait(&full_a[stage], phase);
            mbar_wait(&full_b[stage], phase);
            tc_fence_after();
            uint64_t ad = hi + (uint64_t)(ring_u + (uint32_t)((stage * (kSStage + kSwDy)) >> 4));
            uint64_t bd = ad + (uint64_t)(kSStage >> 4);
#pragma unroll 4
            for (int ks = 0; ks < kSR * kSC / 16; ++ks, ad += 16, bd += 16) {       // 16 consecutive voxels per K step
                if (leader) umma_bf16(tmem_base, ad, bd, idesc, accumulate);
                accumulate = 1;
            }
            if (leader) umma_commit(&empty_bar[stage]);
            __syncwarp();
            if (++stage == kSwStages) { stage = 0; phase ^= 1; }
        }
        if (leader) umma_commit(done_bar);
        __syncwarp();
        FPL_PDL_TRIGGER();
    } else if (warp == 1) {
        // ===================== TMA producer: dy tile [2 groups][16 rows][32 voxels] =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            StemTile c = stem_tile(G, tile_begin);
            for (int t = tile_begin; t < tile_end; ++t, stem_tile_next(G, c)) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                mbar_expect_tx(&full_b[stage], (uint32_t)kSwDy);
                tma_load_5d(ring + stage * (kSStage + kSwDy) + kSStage, &dymap, &full_b[stage], c.w0 * 8, c.h0, P.dy_c8off, c.z, c.n);
                if (++stage == kSwStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp < 6) {
        // ===================== final epilogue: dW[co][tap] += D[tap (hi)] + D[32 + tap (lo)] =====================
        if (tile_end > tile_begin) {
            const int quarter = warp & 3;
            mbar_wait(done_bar, 0);
            tc_fence_after();
            uint32_t r[16];
            tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16), r);
            tmem_ld_wait();
            // M = 64: 16 accumulator rows per 32-lane TMEM quadrant (rows 16 q .. 16 q + 15 in lanes 0..15)
            const int row = quarter * 16 + lane, tap = row & 31;
            if (lane < 16 && tap < 27) {
#pragma unroll
                for (int co = 0; co < 16; ++co) atomicAdd(P.dw + co * 27 + tap, __uint_as_float(r[co]));
            }
        }
    } else {
        // ===================== builders =====================
        const int b = threadIdx.x - 32 * 6;
        STEM_BUILDER_LOOP(stage * (kSStage + kSwDy), full_a, kSwStages)
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 32u);
    }
}

StemGeo stem_geo(int n, int d, int h, int w) {
    StemGeo G;
    G.N = n; G.D = d; G.H = h; G.W = w;
    G.tiles_h = (h + kSR - 1) / kSR; G.tiles_w = (w + kSC - 1) / kSC;
    G.total_tiles = G.tiles_h * G.tiles_w * n * d;
    return G;
}

}  // namespace

bool fpl_stem_tc_eligible(int n, int cin, int d, int h, int w, int cout, int kd) {
    return cin == 1 && cout == 16 && kd == 3 && w >= 32 && h >= 4 && (int64_t)n * d * ((h + 15) / 16) * ((w + 31) / 32) < (1 << 30);
}

int fpl_stem_fwd_tc_launch(const float* x, const float* w, const float* bias, void* y, int y_c8tot, int y_c8off, double* stats, int n,
                           int d, int h, int w_, void* stream) {
    StemFwdParams P;
    P.img = x; P.w = w; P.bias = bias; P.y = (bf16x8*)y; P.stats = stats; P.y_c8tot = y_c8tot; P.y_c8off = y_c8off;
    P.G = stem_geo(n, d, h, w_);
    const int smem_bytes = kSfStages * kSStage + 6 * 512 + 2 * kSHalo * 4 + 256 + 1024;
    int grid = FPL_NUM_SMS;
    if (grid > P.G.total_tiles) grid = P.G.total_tiles;
    FPL_CHECK_CUDA(cudaFuncSetAttribute(stem_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    fpl_launch(stem_fwd_tc_kernel, grid, kSfThreads, smem_bytes, (cudaStream_t)stream, P);
    return 0;
}

int fpl_stem_wgrad_tc_launch(const float* x, const void* dy, int dy_c8tot, int dy_c8off, float* dw, int n, int d, int h, int w_,
                             void* stream) {
    StemWgParams P;
    P.img = x; P.dw = dw; P.dy_c8off = dy_c8off;
    P.G = stem_geo(n, d, h, w_);
    P.split = FPL_NUM_SMS < P.G.total_tiles ? FPL_NUM_SMS : P.G.total_tiles;
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(dy) & 15) == 0, "fpl_stem_conv_wgrad: dy must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_stem_conv_wgrad: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap dymap;
    cuuint64_t gdim[5] = {(cuuint64_t)w_ * 8, (cuuint64_t)h, (cuuint64_t)dy_c8tot, (cuuint64_t)d, (cuuint64_t)n};
    cuuint64_t gstr[4] = {(cuuint64_t)w_ * 16, (cuuint64_t)h * w_ * 16, (cuuint64_t)dy_c8tot * h * w_ * 16,
                          (cuuint64_t)d * dy_c8tot * h * w_ * 16};
    cuuint32_t box[5] = {(cuuint32_t)kSC * 8, (cuuint32_t)kSR, 2, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&dymap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(dy), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_stem_conv_wgrad: cuTensorMapEncodeTiled failed (%d)", (int)r);
    const int smem_bytes = kSwStages * (kSStage + kSwDy) + 2 * kSHalo * 4 + 256 + 1024;
    FPL_CHECK_CUDA(cudaFuncSetAttribute(stem_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    fpl_launch(stem_wgrad_tc_kernel, P.split, kSwThreads, smem_bytes, (cudaStream_t)stream, dymap, P);
    return 0;
}

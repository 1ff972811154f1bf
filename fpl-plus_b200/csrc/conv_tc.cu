// Implicit-GEMM 3-D convolution on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM),
// operands staged by TMA.  Forward and dgrad of nn.Conv3d k(kd,3,3) stride 1 "same" padding
// (PyMIC/pymic/net/net3d/unet2d5_dsbn.py:75,79 and their autograd), bf16 in / fp32 accumulate.
//
// GEMM view per tile:  D[128 voxels x NB] += A[128 x 16] * B[16 x NB]   for every tap and 16-channel slice
//   * tile = 16(H) x 8(W) output voxels of one (n, d) plane; M row r <-> (h0 + r/8, w0 + r%8).
//   * activations are C8-planar ([N][D][C/8][H][W][8] bf16).  One TMA box {80 elem, 18 rows, KC/8 planes}
//     lands a halo'd plane chunk in shared memory as [c8][18][10][8]: that is simultaneously the
//     canonical no-swizzle K-major UMMA layout (8 voxels x 16 B core matrices; SBO = one tile row =
//     160 B, LBO = one channel-group plane = 2880 B), so each of the 9 in-plane taps is the SAME
//     buffer read through a descriptor whose start address is shifted by (kh*10 + kw)*16 B.
//     Zero padding in H/W comes from TMA out-of-bounds fill; out-of-range depth planes are skipped.
//   * weights are pre-staged (fpl_conv3d_prep_weight) as [slice][cin chunk][kd][tap 9][KC/8][NB][8] bf16,
//     i.e. each pipeline stage's B operand is one contiguous chunk fetched with cp.async.bulk.
//   * warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM alloc), warps 2..5 = epilogue
//     (tcgen05.ld -> +bias -> per-channel sum / sum^2 for BatchNorm -> bf16 -> coalesced 16 B stores).
//     Two TMEM accumulator stages overlap the epilogue of tile i with the MMAs of tile i+1.
#include <cuda.h>

#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kTileH = 16, kTileW = 8;
constexpr int kBoxH = kTileH + 2, kBoxW = kTileW + 2;
constexpr int kPlaneBytes = kBoxH * kBoxW * 16;       // one channel-group (8 ch) halo plane: 2880 B
constexpr int kMaxStages = 8;
constexpr int kNumThreads = 192;
constexpr int kSmemBudget = 200 * 1024;

struct TcConfig {
    int nb;        // output channels per CTA tile (UMMA N)
    int kc;        // input channels per pipeline stage
    int nslices, nchunks;
    int a_bytes, b_bytes, stage_bytes, stages;
    int tmem_cols;
    int smem_bytes;
};

bool make_config(int cin, int cout, TcConfig& c) {
    if (cin % 16 != 0 || cout % 16 != 0 || cin <= 0 || cout <= 0) return false;
    c.nb = cout;
    if (c.nb > 128) {
        if (cout % 128 == 0) c.nb = 128;
        else if (cout % 64 == 0) c.nb = 64;
        else if (cout % 32 == 0) c.nb = 32;
        else c.nb = 16;
    }
    c.kc = 64;
    while (c.kc > 16 && (c.kc * c.nb > 4096 || cin % c.kc != 0)) c.kc /= 2;
    if (cin % c.kc != 0) return false;
    c.nslices = cout / c.nb;
    c.nchunks = cin / c.kc;
    c.a_bytes = (c.kc / 8) * kPlaneBytes;
    c.b_bytes = 9 * c.kc * c.nb * 2;
    c.stage_bytes = c.a_bytes + c.b_bytes;
    c.stages = kSmemBudget / c.stage_bytes;
    if (c.stages > kMaxStages) c.stages = kMaxStages;
    if (c.stages < 2) return false;
    // small stages: cap at ~100 KB so two CTAs fit on one SM
    while (c.stages > 3 && c.stages * c.stage_bytes > 100 * 1024) --c.stages;
    int cols = 2 * c.nb;
    c.tmem_cols = 32;
    while (c.tmem_cols < cols) c.tmem_cols *= 2;
    c.smem_bytes = c.stages * c.stage_bytes + 1024 /*align*/ + 256 /*barriers*/ + 2 * cout * (int)sizeof(float) + 16;
    return true;
}

struct TcParams {
    const __nv_bfloat16* image;
    const float* bias;
    bf16x8* y;
    int y_c8tot, y_c8off;
    double* stats;
    int N, D, H, W, cin, cout, kd;
    int x_c8tot, x_c8off;
    int nb, kc, nslices, nchunks, a_bytes, b_bytes, stages, tmem_cols;   // nb / nslices / b_bytes: of THIS launch (after nsub)
    int nsub, nb_img, b_bytes_img;   // N split of a staged image slice: nb = nb_img / nsub (few-tile layers: more, smaller CTAs)
    int tiles_h, tiles_w, total_tiles;
    float* logits;        // head mode: fp32 NCDHW output of the first `classes` channels instead of bf16 C8-planar
    int classes;
    EpiAct act;           // act.scale != NULL: inference epilogue (affine + PReLU + dropout) instead of + bias
};

struct TileCoord {
    int n, d, h0, w0, slice;
};

__device__ __forceinline__ TileCoord decode_tile(const TcParams& P, int t) {
    TileCoord c;
    int tw = t % P.tiles_w; t /= P.tiles_w;
    int th = t % P.tiles_h; t /= P.tiles_h;
    c.d = t % P.D; t /= P.D;
    c.n = t % P.N;
    c.slice = t / P.N;
    c.h0 = th * kTileH;
    c.w0 = tw * kTileW;
    return c;
}

__global__ void __launch_bounds__(kNumThreads) conv3d_tc_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                 const __grid_constant__ CUtensorMap imap, TcParams P) {
    extern __shared__ uint8_t smem_raw[];
    // stage ring at 1024-byte alignment, then barriers, the TMEM base slot and the BN partial sums
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int stage_bytes = P.a_bytes + P.b_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * stage_bytes);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kMaxStages;
    uint64_t* tmem_full = bars + 2 * kMaxStages;
    uint64_t* tmem_empty = bars + 2 * kMaxStages + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);
    float* bias_sm = reinterpret_cast<float*>(bars + 2 * kMaxStages + 6);   // [cout], 16-byte aligned

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pad_d = P.kd / 2;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&xmap) : "memory");
        if (P.nsub > 1) asm volatile("prefetch.tensormap [%0];" ::"l"(&imap) : "memory");
        for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 4); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    FPL_PDL_WAIT();      // prologue above overlapped the previous kernel's tail; from here on its results are visible
    float* scale_sm = bias_sm + P.cout;
    const bool fuse_act = P.act.scale != nullptr;
    for (int i = threadIdx.x; i < P.cout; i += kNumThreads) {
        bias_sm[i] = fuse_act ? P.act.shift[i] : (P.bias != nullptr ? P.bias[i] : 0.0f);
        scale_sm[i] = fuse_act ? P.act.scale[i] : 1.0f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
                TileCoord c = decode_tile(P, t);
                for (int q = 0; q < P.nchunks; ++q) {
                    for (int kdi = 0; kdi < P.kd; ++kdi) {
                        int dz = c.d + kdi - pad_d;
                        if (dz < 0 || dz >= P.D) continue;
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        uint8_t* a_dst = smem + (size_t)stage * stage_bytes;
                        uint8_t* b_dst = a_dst + P.a_bytes;
                        mbar_expect_tx(&full_bar[stage], (uint32_t)(P.a_bytes + P.b_bytes));
                        tma_load_3d(a_dst, &xmap, &full_bar[stage], (c.w0 - 1) * 8, c.h0 - 1,
                                    (c.n * P.D + dz) * P.x_c8tot + P.x_c8off + q * (P.kc / 8));
                        if (P.nsub == 1) {
                            const uint8_t* b_src = reinterpret_cast<const uint8_t*>(P.image) +
                                                   ((size_t)(c.slice * P.nchunks + q) * P.kd + kdi) * P.b_bytes;
                            bulk_load(b_dst, b_src, (uint32_t)P.b_bytes, &full_bar[stage]);
                        } else {
                            // this CTA's nb columns out of the nb_img of the staged slice: the image is a 3-D tensor
                            // {nb_img * 16 B, 9 * kc/8 rows, chunks}; one TMA box lands the packed [rows][nb * 16 B] operand
                            const int simg = c.slice / P.nsub, sub = c.slice - simg * P.nsub;
                            tma_load_3d(b_dst, &imap, &full_bar[stage], sub * P.nb * 2, 0, (simg * P.nchunks + q) * P.kd + kdi);
                        }
                        if (++stage == P.stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: the whole warp runs the loop (uniform), one lane issues =====================
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(P.nb >> 3) << 17) | (8u << 24);
        // descriptors = constant high part + (smem byte address >> 4) in the low 14 bits
        const uint64_t a_hi = make_desc(0, kPlaneBytes, kBoxW * 16), b_hi = make_desc(0, P.nb * 16, 128);
        const uint32_t smem_u = smem_u32(smem) >> 4;
        const uint64_t b_tap_step = (uint64_t)((P.kc / 8) * P.nb);        // 16-byte units between taps of B
        const uint64_t b_k_step = (uint64_t)(2 * P.nb);                   // ... between 16-channel K steps
        const int ksteps = P.kc / 16;
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            TileCoord c = decode_tile(P, t);
            mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(acc * P.nb);
            uint32_t accumulate = 0;
            for (int q = 0; q < P.nchunks; ++q) {
                for (int kdi = 0; kdi < P.kd; ++kdi) {
                    int dz = c.d + kdi - pad_d;
                    if (dz < 0 || dz >= P.D) continue;
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t a_base = smem_u + (uint32_t)(((size_t)stage * stage_bytes) >> 4);
                    const uint32_t b_base = a_base + (uint32_t)(P.a_bytes >> 4);
                    // descriptor arithmetic as 64-bit adds of warp-uniform values (the 14-bit start-address field never
                    // carries): stays on the uniform datapath instead of per-thread IMAD / LOP3 + R2UR moves per MMA
                    uint64_t a_j = a_hi + (uint64_t)a_base, b_j = b_hi + (uint64_t)b_base;
                    for (int j = 0; j < ksteps; ++j) {
                        uint64_t bdesc = b_j;
#pragma unroll
                        for (int t9 = 0; t9 < 9; ++t9) {
                            const uint64_t adesc = a_j + (uint64_t)((t9 / 3) * kBoxW + (t9 % 3));
                            if (leader) umma_bf16(d_tmem, adesc, bdesc, idesc, accumulate);
                            accumulate = 1;
                            bdesc += b_tap_step;
                        }
                        a_j += 2 * kPlaneBytes / 16;
                        b_j += b_k_step;
                    }
                    if (leader) umma_commit(&empty_bar[stage]);      // smem slot reusable once these MMAs retire
                    __syncwarp();
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
            }
            if (leader) umma_commit(&tmem_full[acc]);                // accumulator ready for the epilogue
            __syncwarp();
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        FPL_PDL_TRIGGER();   // this CTA has issued its last tile: the next kernel of the stream may be scheduled as SMs drain
    } else {
        // ===================== epilogue (warps 2..5) =====================
        // thread = one output voxel (TMEM lane); per 16-channel chunk: +bias, one 2 x 128-bit bf16 store,
        // and the BatchNorm partial sums through a transposing butterfly (lane L ends up owning channel
        // L of the sum, lane 16+L of the sum of squares).  The per-lane totals stay in registers across
        // all tiles of a slice and reach global memory once per slice (double atomics).
        const int quarter = warp & 3;                        // TMEM lane quarter this warp may access
        const int row = quarter * 32 + lane;
        const int hl = row / kTileW, wl = row % kTileW;
        int acc = 0; uint32_t acc_phase = 0;
        int cur_slice = -1;
        constexpr int kMaxChunks = 8;                        // nb <= 128
        // fp64 across tiles: fp32 running sums over the hundreds of tiles a warp walks at 16 SMs lose enough of sum y^2
        // that var = E[y^2] - mean^2 is off by 2.5e-5 relative at mean/std = 30 (tests/test_gpu_train_kernels.py)
        double run[kMaxChunks];
#pragma unroll
        for (int k = 0; k < kMaxChunks; ++k) run[k] = 0.0;
        const bool want_stats = P.stats != nullptr;
        const int nchunk16 = P.nb / 16;
        const float act_slope = fuse_act ? __ldg(P.act.slope) : 0.0f;
        const float act_keep_scale = (fuse_act && P.act.drop_p > 0.0f) ? 1.0f / (1.0f - P.act.drop_p) : 1.0f;
        const uint64_t act_seed = fuse_act ? P.act.seed + (P.act.seed_dev != nullptr ? (uint64_t)__ldg(P.act.seed_dev) : 0ull) : 0ull;
        for (int t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
            TileCoord c = decode_tile(P, t);
            if (want_stats && c.slice != cur_slice) {
                if (cur_slice >= 0) {
#pragma unroll
                    for (int k = 0; k < kMaxChunks; ++k) {
                        if (k < nchunk16) {
                            atomicAdd(P.stats + (lane >> 4) * P.cout + cur_slice * P.nb + k * 16 + (lane & 15), run[k]);
                            run[k] = 0.0;
                        }
                    }
                }
                cur_slice = c.slice;
            }
            const int h = c.h0 + hl, w = c.w0 + wl;
            const bool valid = h < P.H && w < P.W;
            const int64_t HW = (int64_t)P.H * P.W;
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const int64_t out_base = (((int64_t)c.n * P.D + c.d) * P.y_c8tot + P.y_c8off + (c.slice * P.nb) / 8) * HW +
                                     (int64_t)h * P.W + w;
            const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * P.nb);
#pragma unroll
            for (int k = 0; k < kMaxChunks; ++k) {
                if (k < nchunk16) {
                    const int c0 = k * 16;
                    uint32_t r[16];
                    tmem_ld16(t_row + (uint32_t)c0, r);
                    tmem_ld_wait();
                    float v[32];
                    const float4* b4 = reinterpret_cast<const float4*>(bias_sm + c.slice * P.nb + c0);
                    if (!fuse_act) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            float4 bb = b4[i];
                            v[4 * i + 0] = __uint_as_float(r[4 * i + 0]) + bb.x;
                            v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + bb.y;
                            v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + bb.z;
                            v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + bb.w;
                        }
                    } else {
                        // inference: BatchNorm (running statistics) + PReLU + dropout applied here, the activation kernel
                        // and its extra pass over the tensor disappear
                        const float4* s4 = reinterpret_cast<const float4*>(scale_sm + c.slice * P.nb + c0);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 bb = b4[i], ss = s4[i];
                            const float sc[4] = {ss.x, ss.y, ss.z, ss.w}, sh[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float z = fmaf(__uint_as_float(r[4 * i + q]), sc[q], sh[q]);
                                v[4 * i + q] = z > 0.0f ? z : act_slope * z;
                            }
                        }
                        if (P.act.drop_p > 0.0f && valid) {
                            const int C8 = P.cout >> 3;
                            const int64_t vec0 = (((int64_t)c.n * P.D + c.d) * C8 + (c.slice * P.nb + c0) / 8) * HW + (int64_t)h * P.W + w;
#pragma unroll
                            for (int g = 0; g < 2; ++g) {
                                const uint32_t keep = dropout_keep8(act_seed, P.act.offset, (uint64_t)(vec0 + (int64_t)g * HW), P.act.drop_p);
#pragma unroll
                                for (int i = 0; i < 8; ++i) v[8 * g + i] = ((keep >> i) & 1u) ? v[8 * g + i] * act_keep_scale : 0.0f;
                            }
                        }
                    }
                    if (P.logits != nullptr) {
                        if (valid && k == 0) {
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                if (i < P.classes)
                                    P.logits[(((int64_t)c.n * P.classes + i) * P.D + c.d) * HW + (int64_t)h * P.W + w] = v[i];
                        }
                    } else if (valid) {
                        st_bf16x8(P.y + out_base + (int64_t)(c0 / 8) * HW, v);
                        st_bf16x8(P.y + out_base + (int64_t)(c0 / 8 + 1) * HW, v + 8);
                    }
                    if (want_stats) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            v[i] = valid ? v[i] : 0.0f;
                            v[16 + i] = v[i] * v[i];
                        }
                        warp_transpose_sum32(v, lane);
                        run[k] += (double)v[0];
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (want_stats && cur_slice >= 0) {
#pragma unroll
            for (int k = 0; k < kMaxChunks; ++k)
                if (k < nchunk16)
                    atomicAdd(P.stats + (lane >> 4) * P.cout + cur_slice * P.nb + k * 16 + (lane & 15), run[k]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
    }
}

// ---------------------------------------------------------------------------------------------
// weight staging: fp32 [Cout][Cin][T] -> bf16 [slice][chunk][kd][tap9][KC/8][NB][8]
// ---------------------------------------------------------------------------------------------
__global__ void prep_weight_kernel(const float* __restrict__ w, __nv_bfloat16* image, int cin_eff, int cout_eff, int kd,
                                   int transpose_flip, int nb, int kc, int64_t total) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int T = kd * 9;
    const int nchunks = cin_eff / kc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t t = i;
        int e = (int)(t % 8); t /= 8;
        int nrow = (int)(t % nb); t /= nb;
        int k8 = (int)(t % (kc / 8)); t /= (kc / 8);
        int t9 = (int)(t % 9); t /= 9;
        int kdi = (int)(t % kd); t /= kd;
        int q = (int)(t % nchunks);
        int s = (int)(t / nchunks);
        int out = s * nb + nrow, in = q * kc + k8 * 8 + e, tap = kdi * 9 + t9;
        float v;
        if (!transpose_flip) v = w[((int64_t)out * cin_eff + in) * T + tap];
        else v = w[((int64_t)in * cout_eff + out) * T + (T - 1 - tap)];   // w is [Cout_fwd = cin_eff][Cin_fwd = cout_eff][T]
        image[i] = __float2bfloat16_rn(v);
    }
}

}  // namespace

extern "C" int64_t fpl_conv3d_weight_image_bytes(int cin, int cout, int kd) {
    TcConfig c;
    if (!make_config(cin, cout, c)) return -1;
    return (int64_t)c.nslices * c.nchunks * kd * c.b_bytes;
}

extern "C" int fpl_conv3d_prep_weight(const float* w, int cin, int cout, int kd, int transpose_flip, void* image,
                                      void* stream) {
    const int cin_eff = transpose_flip ? cout : cin, cout_eff = transpose_flip ? cin : cout;
    TcConfig c;
    FPL_REQUIRE(make_config(cin_eff, cout_eff, c), "fpl_conv3d_prep_weight: unsupported channels (%d -> %d)", cin_eff, cout_eff);
    FPL_REQUIRE(kd == 1 || kd == 3, "fpl_conv3d_prep_weight: kd=%d must be 1 or 3", kd);
    int64_t total = (int64_t)c.nslices * c.nchunks * kd * c.b_bytes / 2;
    int blocks = (int)((total + 255) / 256);
    if (blocks > FPL_NUM_SMS * 8) blocks = FPL_NUM_SMS * 8;
    fpl_launch(prep_weight_kernel, blocks, 256, 0, (cudaStream_t)stream, w, (__nv_bfloat16*)image, cin_eff, cout_eff, kd,
                                                                 transpose_flip, c.nb, c.kc, total);
    FPL_LAUNCH_CHECK();
    return 0;
}

// all weight images of a network in ONE launch (blockIdx.y = conv): the per-step refresh after the
// optimiser update costs one launch instead of one per conv and direction
constexpr int kMaxPrepBatch = 80;
struct PrepBatch {
    const float* w[kMaxPrepBatch];
    __nv_bfloat16* image[kMaxPrepBatch];
    int cin_eff[kMaxPrepBatch], cout_eff[kMaxPrepBatch];
    unsigned char kd[kMaxPrepBatch], tf[kMaxPrepBatch];
    short nb[kMaxPrepBatch], kc[kMaxPrepBatch];
    int total[kMaxPrepBatch];
};

namespace {
// One thread per (output channel, input channel) PAIR: it reads the pair's kd*9 taps as one contiguous run of the PyTorch
// layout (108 B for k3: whole sectors) and writes them to the kd*9 tap planes of the image; consecutive threads are
// consecutive image elements of a tap plane, so every warp store is one 64-byte run.  (The element-per-thread form
// of prep_weight_kernel costs 7 integer divisions and one 32-byte sector per 4-byte read: 112 us per step for the 36
// images of the network, at the head of every optimiser step.)
__global__ void prep_weight_batch_kernel(const __grid_constant__ PrepBatch B) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int e = blockIdx.y;
    const float* __restrict__ w = B.w[e];
    __nv_bfloat16* image = B.image[e];
    const int cin_eff = B.cin_eff[e], cout_eff = B.cout_eff[e], kd = B.kd[e], nb = B.nb[e], kc = B.kc[e];
    const int T = kd * 9, nchunks = cin_eff / kc;
    const int plane = (kc / 8) * nb * 8;                  // elements of one tap plane of one (slice, chunk)
    const int pairs = cin_eff * cout_eff;
    const bool tf = B.tf[e] != 0;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < pairs; r += gridDim.x * blockDim.x) {
        const int sq = r / plane, rem = r - sq * plane;   // (slice, chunk) and position inside a tap plane
        const int el = rem & 7, nrow = (rem >> 3) % nb, k8 = (rem >> 3) / nb;
        const int q = sq % nchunks, sl = sq / nchunks;
        const int out = sl * nb + nrow, in = q * kc + k8 * 8 + el;
        const float* src = tf ? w + ((int64_t)in * cout_eff + out) * T : w + ((int64_t)out * cin_eff + in) * T;
        __nv_bfloat16* dst = image + (int64_t)sq * T * plane + rem;
        if (kd == 3) {
#pragma unroll
            for (int tap = 0; tap < 27; ++tap) dst[(int64_t)tap * plane] = __float2bfloat16_rn(__ldg(src + (tf ? 26 - tap : tap)));
        } else {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) dst[(int64_t)tap * plane] = __float2bfloat16_rn(__ldg(src + (tf ? 8 - tap : tap)));
        }
    }
}
}  // namespace

extern "C" int fpl_conv3d_prep_weight_batch(int count, const float* const* h_w, const int* h_cin, const int* h_cout,
                                            const int* h_kd, const int* h_transpose_flip, void* const* h_images,
                                            void* stream) {
    FPL_REQUIRE(count >= 0 && count <= kMaxPrepBatch, "fpl_conv3d_prep_weight_batch: count %d not in [0,%d]", count, kMaxPrepBatch);
    if (count == 0) return 0;
    PrepBatch B;
    int max_total = 0;
    for (int e = 0; e < count; ++e) {
        const int tf = h_transpose_flip[e];
        const int cin_eff = tf ? h_cout[e] : h_cin[e], cout_eff = tf ? h_cin[e] : h_cout[e];
        TcConfig c;
        FPL_REQUIRE(make_config(cin_eff, cout_eff, c), "fpl_conv3d_prep_weight_batch: unsupported channels (%d -> %d)", cin_eff, cout_eff);
        FPL_REQUIRE(h_kd[e] == 1 || h_kd[e] == 3, "fpl_conv3d_prep_weight_batch: kd=%d must be 1 or 3", h_kd[e]);
        B.w[e] = h_w[e]; B.image[e] = (__nv_bfloat16*)h_images[e];
        B.cin_eff[e] = cin_eff; B.cout_eff[e] = cout_eff; B.kd[e] = (unsigned char)h_kd[e]; B.tf[e] = (unsigned char)tf;
        B.nb[e] = (short)c.nb; B.kc[e] = (short)c.kc;
        B.total[e] = c.nslices * c.nchunks * h_kd[e] * c.b_bytes / 2;
        if (B.total[e] > max_total) max_total = B.total[e];
    }
    // one thread per (out, in) pair of the largest layer (65 536 pairs at 256 -> 256); blocks beyond a small layer's
    // pair count exit at once
    int bx = (max_total / 9 + 255) / 256;
    if (bx > 512) bx = 512;
    if (bx < 1) bx = 1;
    fpl_launch(prep_weight_batch_kernel, dim3(bx, count), 256, 0, (cudaStream_t)stream, B);
    FPL_LAUNCH_CHECK();
    return 0;
}

static int conv3d_tc_launch(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias, void* y,
                            int y_c8tot, int y_c8off, double* stats, int n, int d, int h, int w, int cin, int cout,
                            int kd, float* logits, int classes, void* stream, const EpiAct* act = nullptr) {
    TcConfig c;
    FPL_REQUIRE(make_config(cin, cout, c), "fpl_conv3d_tc: unsupported channels (%d -> %d); need multiples of 16", cin, cout);
    FPL_REQUIRE(kd == 1 || kd == 3, "fpl_conv3d_tc: kd=%d must be 1 or 3", kd);
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(image) & 15) == 0,
                "fpl_conv3d_tc: x/image must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_conv3d_tc: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap xmap;
    cuuint64_t gdim[3] = {(cuuint64_t)w * 8, (cuuint64_t)h, (cuuint64_t)n * d * x_c8tot};
    cuuint64_t gstride[2] = {(cuuint64_t)w * 16, (cuuint64_t)h * w * 16};
    cuuint32_t box[3] = {(cuuint32_t)kBoxW * 8, (cuuint32_t)kBoxH, (cuuint32_t)(c.kc / 8)};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = encode(&xmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(x), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_tc: cuTensorMapEncodeTiled failed (%d) for dims [%d,%d,%d] c8tot=%d", (int)r,
                w * 8, h, n * d * x_c8tot, x_c8tot);
    TcParams P;
    P.image = (const __nv_bfloat16*)image; P.bias = bias; P.y = (bf16x8*)y; P.y_c8tot = y_c8tot; P.y_c8off = y_c8off;
    P.stats = stats; P.N = n; P.D = d; P.H = h; P.W = w; P.cin = cin; P.cout = cout; P.kd = kd;
    P.x_c8tot = x_c8tot; P.x_c8off = x_c8off;
    P.nb = c.nb; P.kc = c.kc; P.nslices = c.nslices; P.nchunks = c.nchunks; P.a_bytes = c.a_bytes; P.b_bytes = c.b_bytes;
    P.stages = c.stages; P.tmem_cols = c.tmem_cols;
    P.tiles_h = (h + kTileH - 1) / kTileH; P.tiles_w = (w + kTileW - 1) / kTileW;
    // few voxel tiles (levels 3-4): split the N of a staged slice over up to 4 CTAs so that the ~430 serial MMAs of a tile
    // get shorter and more SMs work; the image layout stays that of nb_img
    P.nsub = 1; P.nb_img = c.nb; P.b_bytes_img = c.b_bytes;
    {
        const int64_t mn = (int64_t)P.tiles_h * P.tiles_w * d * n * c.nslices;
        while (logits == nullptr && P.nsub < 4 && c.nb % (P.nsub * 2 * 16) == 0 && c.nb / (P.nsub * 2) >= 32 &&
               mn * P.nsub < 96)
            P.nsub *= 2;
    }
    P.nb = c.nb / P.nsub; P.nslices = c.nslices * P.nsub; P.b_bytes = c.b_bytes / P.nsub;
    int64_t total = (int64_t)P.tiles_h * P.tiles_w * d * n * P.nslices;
    FPL_REQUIRE(total < (1ll << 30), "fpl_conv3d_tc: too many tiles");
    P.total_tiles = (int)total;
    P.logits = logits; P.classes = classes;
    if (act != nullptr) P.act = *act; else { P.act.scale = nullptr; P.act.shift = nullptr; P.act.slope = nullptr; P.act.drop_p = 0.0f; P.act.seed = P.act.offset = 0; P.act.seed_dev = nullptr; }
    FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, c.smem_bytes));
    int ctas_per_sm = c.smem_bytes <= 110 * 1024 ? 2 : 1;
    int grid = FPL_NUM_SMS * ctas_per_sm;
    if (grid > P.total_tiles) grid = P.total_tiles;
    CUtensorMap imap = xmap;
    if (P.nsub > 1) {
        // 8-byte elements: nb * 16 B = nb * 2 elements (<= 256 per box dimension)
        const int rows = 9 * (c.kc / 8);
        cuuint64_t idim[3] = {(cuuint64_t)c.nb * 2, (cuuint64_t)rows, (cuuint64_t)c.nslices * c.nchunks * kd};
        cuuint64_t istride[2] = {(cuuint64_t)c.nb * 16, (cuuint64_t)c.b_bytes};
        cuuint32_t ibox[3] = {(cuuint32_t)P.nb * 2, (cuuint32_t)rows, 1};
        r = encode(&imap, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<void*>(image), idim, istride, ibox, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_tc: cuTensorMapEncodeTiled (weight image) failed (%d)", (int)r);
    }
    fpl_launch(conv3d_tc_kernel, grid, kNumThreads, c.smem_bytes, (cudaStream_t)stream, xmap, imap, P);
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_conv3d_tc(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias, void* y,
                             int y_c8tot, int y_c8off, double* stats, int n, int d, int h, int w, int cin, int cout,
                             int kd, void* stream) {
    return conv3d_tc_launch(x, x_c8tot, x_c8off, image, bias, y, y_c8tot, y_c8off, stats, n, d, h, w, cin, cout, kd,
                            nullptr, 0, stream);
}

/* Inference form of fpl_conv3d_tc: the epilogue applies a = dropout(prelu(acc * scale + shift)) (eval-mode BatchNorm,
 * nn.PReLU, nn.Dropout of unet2d5_dsbn.py:75-81) and writes the ACTIVATION, so no fpl_dsbn_act_fwd pass follows. */
extern "C" int fpl_conv3d_tc_act(const void* x, int x_c8tot, int x_c8off, const void* image, void* a, int a_c8tot, int a_c8off,
                                 int n, int d, int h, int w, int cin, int cout, int kd, const float* scale, const float* shift,
                                 const float* slope, float drop_p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                                 void* stream) {
    FPL_REQUIRE(scale != nullptr && shift != nullptr && slope != nullptr, "fpl_conv3d_tc_act: scale/shift/slope required");
    FPL_REQUIRE(drop_p >= 0.0f && drop_p < 1.0f, "fpl_conv3d_tc_act: dropout p=%f out of [0,1)", drop_p);
    EpiAct act;
    act.scale = scale; act.shift = shift; act.slope = slope; act.drop_p = drop_p; act.seed = seed; act.offset = offset;
    act.seed_dev = (const unsigned long long*)seed_dev;
    return conv3d_tc_launch(x, x_c8tot, x_c8off, image, nullptr, a, a_c8tot, a_c8off, nullptr, n, d, h, w, cin, cout, kd,
                            nullptr, 0, stream, &act);
}

extern "C" int fpl_head_conv_tc(const void* x, int x_c8tot, int x_c8off, const void* image16, const float* bias16,
                                float* logits, int n, int d, int h, int w, int cin, int classes, void* stream) {
    FPL_REQUIRE(classes >= 1 && classes <= 8, "fpl_head_conv_tc: class_num=%d not in [1,8]", classes);
    FPL_REQUIRE(logits != nullptr, "fpl_head_conv_tc: logits required");
    return conv3d_tc_launch(x, x_c8tot, x_c8off, image16, bias16, nullptr, 0, 0, nullptr, n, d, h, w, cin, 16, 1, logits,
                            classes, stream);
}

// DSBN BatchNorm3d + PReLU + Dropout + MaxPool, forward and backward, on C8-planar bf16.
// Replaces nn.BatchNorm3d (selected domain, net_run_dsbn/dsbn.py:54-57), nn.PReLU,
// nn.Dropout and nn.MaxPool3d of PyMIC/pymic/net/net3d/unet2d5_dsbn.py:75-81,104-117.
// All kernels are HBM-streaming: one 16-byte vector (8 channels of one voxel) per access,
// consecutive threads on consecutive voxels of one (n, d, channel-group) plane.
#include "common.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------
// finalize: batch statistics -> scale/shift, running statistics update
// ------------------------------------------------------------------------------------
__global__ void dsbn_finalize_kernel(const double* __restrict__ stats, double inv_count, double unbias,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* running_mean, float* running_var, long long* nbt,
                                     float momentum, float eps, int training,
                                     float* scale, float* shift, float* save_mean, float* save_invstd, int C) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < C) {
        float mean, invstd;
        if (training) {
            double m = stats[c] * inv_count;
            double var = stats[C + c] * inv_count - m * m;
            if (var < 0.0) var = 0.0;
            mean = (float)m;
            invstd = (float)(1.0 / sqrt(var + (double)eps));
            if (running_mean != nullptr) {
                running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * mean;
                running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)(var * unbias);
            }
        } else {
            mean = running_mean[c];
            invstd = rsqrtf(running_var[c] + eps);
            invstd = 1.0f / sqrtf(running_var[c] + eps);
        }
        float g = gamma[c] * invstd;
        scale[c] = g;
        shift[c] = beta[c] - mean * g;
        save_mean[c] = mean;
        save_invstd[c] = invstd;
    }
    if (training && nbt != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *nbt += 1;
}

// ------------------------------------------------------------------------------------
// forward: a = dropout(prelu(y*scale+shift)), optional fused max-pool
// ------------------------------------------------------------------------------------
// optional fused "finalize" (statistics -> scale/shift, running-stat update) executed in the prologue of
// the activation kernels: every block derives the affine map of ITS 8 channels, one block per channel
// group publishes it (for backward) and updates the selected domain's running statistics
struct BnFinalize {
    const double* stats;        // non-NULL (training) or running_mean non-NULL (eval) enables the fused path
    double inv_count, unbias;
    const float* gamma;
    const float* beta;
    float* running_mean;
    float* running_var;
    long long* nbt;
    float momentum, eps;
    int training, enabled;
    float* scale;
    float* shift;
    float* save_mean;
    float* save_invstd;
};

struct ActParams {
    BnFinalize fin;
    const bf16x8* y;            // dense [N][D][C8][H][W]
    const float* scale;
    const float* shift;
    const float* slope;
    bf16x8* a;
    int a_c8tot, a_c8off;
    bf16x8* pooled;
    int p_c8tot, p_c8off;
    uint2* pool_idx;            // 8 x uint8 per pooled vector
    int pool_kd;
    float drop_p;
    const uint2* drop_mask;     // 8 x uint8 per vector, dense order
    uint64_t seed, offset;
    const unsigned long long* seed_dev;   // optional device-side addend to the seed (CUDA-graph replays)
    int N, D, C8, H, W;
};

__device__ __forceinline__ void load_affine(const float* scale, const float* shift, int c8, float* sc, float* sh) {
    const float4* s4 = reinterpret_cast<const float4*>(scale + c8 * 8);
    const float4* h4 = reinterpret_cast<const float4*>(shift + c8 * 8);
    float4 a = __ldg(s4), b = __ldg(s4 + 1), c = __ldg(h4), d = __ldg(h4 + 1);
    sc[0] = a.x; sc[1] = a.y; sc[2] = a.z; sc[3] = a.w; sc[4] = b.x; sc[5] = b.y; sc[6] = b.z; sc[7] = b.w;
    sh[0] = c.x; sh[1] = c.y; sh[2] = c.z; sh[3] = c.w; sh[4] = d.x; sh[5] = d.y; sh[6] = d.z; sh[7] = d.w;
}

__device__ __forceinline__ void bn_prologue(const BnFinalize& F, int C, int c8, bool writer, float* sc, float* sh) {
    __shared__ float s_aff[16];
    if (threadIdx.x < 8) {
        const int c = c8 * 8 + threadIdx.x;
        float mean, invstd;
        if (F.training) {
            double m = F.stats[c] * F.inv_count;
            double var = F.stats[C + c] * F.inv_count - m * m;
            if (var < 0.0) var = 0.0;
            mean = (float)m;
            invstd = (float)(1.0 / sqrt(var + (double)F.eps));
            if (writer && F.running_mean != nullptr) {
                F.running_mean[c] = (1.0f - F.momentum) * F.running_mean[c] + F.momentum * mean;
                F.running_var[c] = (1.0f - F.momentum) * F.running_var[c] + F.momentum * (float)(var * F.unbias);
            }
        } else {
            mean = F.running_mean[c];
            invstd = 1.0f / sqrtf(F.running_var[c] + F.eps);
        }
        const float g = F.gamma[c] * invstd;
        s_aff[threadIdx.x] = g;
        s_aff[8 + threadIdx.x] = F.beta[c] - mean * g;
        if (writer) {
            F.scale[c] = g;
            F.shift[c] = F.beta[c] - mean * g;
            F.save_mean[c] = mean;
            F.save_invstd[c] = invstd;
            if (c == 0 && F.training && F.nbt != nullptr) *F.nbt += 1;
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) { sc[i] = s_aff[i]; sh[i] = s_aff[8 + i]; }
}

__device__ __forceinline__ uint32_t keep_bits(const uint2* mask, uint64_t seed, uint64_t offset, int64_t vec, float p) {
    if (mask != nullptr) {
        uint2 m = __ldg(mask + vec);
        uint32_t bits = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            bits |= (((m.x >> (8 * i)) & 0xffu) ? 1u : 0u) << i;
            bits |= (((m.y >> (8 * i)) & 0xffu) ? 1u : 0u) << (4 + i);
        }
        return bits;
    }
    return dropout_keep8(seed, offset, (uint64_t)vec, p);
}

// grid: (blocks per channel group, C8).  A block stays inside one channel group (its affine parameters, derived once in
// the prologue, live in registers) and walks over work items = (plane (n,d), chunk of 2*256 vectors), two vectors per
// thread in flight, with stepped plane pointers (same structure as dsbn_act_bwd_kernel below).
__global__ void __launch_bounds__(kThreads) dsbn_act_fwd_kernel(const __grid_constant__ ActParams P) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int HW = P.H * P.W;
    const int c8 = blockIdx.y;
    const float slope = __ldg(P.slope);
    const bool drop = P.drop_p > 0.0f;
    const float keep_scale = drop ? 1.0f / (1.0f - P.drop_p) : 1.0f;
    const uint64_t seed = P.seed + (P.seed_dev != nullptr ? (uint64_t)__ldg(P.seed_dev) : 0ull);
    float sc[8], sh[8];
    if (P.fin.enabled) bn_prologue(P.fin, P.C8 * 8, c8, blockIdx.x == 0, sc, sh);
    else load_affine(P.scale, P.shift, c8, sc, sh);
    const int chunks = (HW + 2 * kThreads - 1) / (2 * kThreads);
    const int items = P.N * P.D * chunks;
    const int step_nd = gridDim.x / chunks, step_ch = gridDim.x - step_nd * chunks;
    int nd = blockIdx.x / chunks, ch = blockIdx.x - nd * chunks;
    const int64_t y_stride = (int64_t)P.C8 * HW, a_stride = (int64_t)P.a_c8tot * HW;
    const bf16x8* src = P.y + ((int64_t)nd * P.C8 + c8) * HW + threadIdx.x;
    bf16x8* dst = P.a + ((int64_t)nd * P.a_c8tot + P.a_c8off + c8) * HW + threadIdx.x;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int voff = ch * (2 * kThreads);
        const int hw = voff + (int)threadIdx.x, hw2 = hw + kThreads;
        const bool one = hw < HW, two = hw2 < HW;
        int4 r0 = make_int4(0, 0, 0, 0), r1 = make_int4(0, 0, 0, 0);
        if (one) r0 = ld_stream16(src + voff);
        if (two) r1 = ld_stream16(src + voff + kThreads);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (!(k == 0 ? one : two)) continue;
            float f[8];
            bf16x8_to_float(*reinterpret_cast<bf16x8*>(k == 0 ? &r0 : &r1), f);
            uint32_t keep = 0xffu;
            if (drop) keep = keep_bits(P.drop_mask, seed, P.offset, (src - P.y) + voff + k * kThreads, P.drop_p);   // dense index of this vector
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float z = fmaf(f[i], sc[i], sh[i]);
                float a = z > 0.0f ? z : slope * z;
                f[i] = ((keep >> i) & 1u) ? a * keep_scale : 0.0f;
            }
            st_bf16x8(dst + voff + k * kThreads, f);
        }
        int dnd = step_nd;
        ch += step_ch;
        if (ch >= chunks) { ch -= chunks; ++dnd; }
        src += dnd * y_stride;
        dst += dnd * a_stride;
    }
}

// one thread per pooled output vector; reads the 2x2x2 (or 1x2x2) window, writes the full
// resolution activations, the pooled max and the 3-bit argmax code (first max wins, scan
// order d,h,w as in torch's max_pool3d).
// grid: (blocks per channel group, C8); work items = (pooled plane (n,d2), chunk of 256 pooled vectors)
__global__ void __launch_bounds__(kThreads) dsbn_act_pool_fwd_kernel(const __grid_constant__ ActParams P) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int kd = P.pool_kd;
    const int D2 = P.D / kd, H2 = P.H / 2, W2 = P.W / 2;
    const int HW = P.H * P.W, HW2 = H2 * W2;
    const int c8 = blockIdx.y;
    const float slope = __ldg(P.slope);
    float sc[8], sh[8];
    if (P.fin.enabled) bn_prologue(P.fin, P.C8 * 8, c8, blockIdx.x == 0, sc, sh);
    else load_affine(P.scale, P.shift, c8, sc, sh);
    const int chunks = (HW2 + kThreads - 1) / kThreads;
    const int items = P.N * D2 * chunks;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int nd2 = item / chunks;
        const int v = (item - nd2 * chunks) * kThreads + (int)threadIdx.x;
        if (v >= HW2) continue;
        const int n = nd2 / D2, d2 = nd2 - n * D2;
        const int h2 = v / W2, w2 = v - h2 * W2;
        float best[8];
        uint32_t code[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { best[i] = -INFINITY; code[i] = 0; }
        int4 raw[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {                      // all loads of the 2x2x2 window first
            const int dd = q >> 2, hh = (q >> 1) & 1, ww = q & 1;
            if (dd < kd) {
                const int64_t nd = (int64_t)n * P.D + d2 * kd + dd;
                raw[q] = ld_stream16(P.y + (nd * P.C8 + c8) * HW + (h2 * 2 + hh) * P.W + w2 * 2 + ww);
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int dd = q >> 2, hh = (q >> 1) & 1, ww = q & 1;
            if (dd < kd) {
                const int64_t nd = (int64_t)n * P.D + d2 * kd + dd;
                float f[8];
                bf16x8_to_float(*reinterpret_cast<bf16x8*>(&raw[q]), f);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float z = fmaf(f[i], sc[i], sh[i]);
                    f[i] = z > 0.0f ? z : slope * z;
                }
                bf16x8 outv = float_to_bf16x8(f);
                st_bf16x8(P.a + (nd * P.a_c8tot + P.a_c8off + c8) * HW + (h2 * 2 + hh) * P.W + w2 * 2 + ww, f);
                // compare on the bf16-rounded values (what backward and the next layer see); first max wins
                bf16x8_to_float(outv, f);
                const uint32_t k = (uint32_t)((dd * 2 + hh) * 2 + ww);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (f[i] > best[i]) { best[i] = f[i]; code[i] = k; }
                }
            }
        }
        st_bf16x8(P.pooled + ((int64_t)nd2 * P.p_c8tot + P.p_c8off + c8) * HW2 + v, best);
        uint2 packed;
        packed.x = code[0] | (code[1] << 8) | (code[2] << 16) | (code[3] << 24);
        packed.y = code[4] | (code[5] << 8) | (code[6] << 16) | (code[7] << 24);
        P.pool_idx[((int64_t)nd2 * P.C8 + c8) * HW2 + v] = packed;
    }
}

// ------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------
struct ActBwdParams {
    const bf16x8* y;
    const bf16x8* g1;
    int g1_c8tot, g1_c8off;
    const bf16x8* g_pool;
    int gp_c8tot, gp_c8off;
    const uint2* pool_idx;
    int pool_kd;
    const float* scale;
    const float* shift;
    const float* mean;
    const float* invstd;
    const float* slope;
    float drop_p;
    const uint2* drop_mask;
    uint64_t seed, offset;
    const unsigned long long* seed_dev;
    double* red;                // [2C+1]: sum dz, sum dz*xhat, dslope
    float* fin_dgamma;          // optional fused finalize of the apply pass (all may be NULL)
    float* fin_dbeta;
    float* fin_dslope;
    float* fin_dbias;
    bf16x8* dy;
    int training;
    double inv_count;
    int N, D, C8, H, W;
    int w_shift;                // log2(W) when W is a power of two, else -1
};

// grid: (blocks per channel group, C8).  A block stays inside one channel group (its per-channel constants live in
// registers) and walks over work items = (plane (n,d), chunk of kBwdV*256 vectors of that plane), kBwdV vectors per thread
// in flight.  The reduce pass ends with ONE block reduction + 17 double atomics per block (a few hundred blocks per
// launch, not one per 1024 vectors: same-address atomics would otherwise serialise at L2).
//   reduce: accumulates sum dz, sum dz*y (raw conv output; turned into sum dz*xhat per block in double) and dslope
//   apply : dy = sc*(dz - m1 - xhat*m2)  rewritten as  sc*dz + cb + cy*y  (cb, cy per channel)
// __launch_bounds__(256, 4): <= 64 registers, 1024 threads per SM keep >= 64 KB of loads in flight.
constexpr int kBwdV = 2;                  // vectors per thread per work item
constexpr int kBwdBlocks = 4;             // resident blocks per SM the register budget is tuned for
template <bool APPLY, bool POOL, bool DROP>
__global__ void __launch_bounds__(kThreads, kBwdBlocks) dsbn_act_bwd_kernel(const __grid_constant__ ActBwdParams P) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int HW = P.H * P.W;
    const int c8 = blockIdx.y;
    const int C = P.C8 * 8;
    const float slope = __ldg(P.slope);
    const float keep_scale = DROP ? 1.0f / (1.0f - P.drop_p) : 1.0f;
    uint64_t seed = 0;
    if (DROP) seed = P.seed + (P.seed_dev != nullptr ? (uint64_t)__ldg(P.seed_dev) : 0ull);
    float sc[8], sh[8];
    load_affine(P.scale, P.shift, c8, sc, sh);
    float ka[8], kb[8];          // reduce: s1, s2 accumulators; apply: cb, cy
    float dsl = 0.0f;
    if (APPLY) {
        if (blockIdx.x == 0 && threadIdx.x < 8) {
            // one block per channel group publishes the parameter gradients (what fpl_dsbn_bwd_finalize does)
            const int c = c8 * 8 + threadIdx.x;
            if (P.fin_dbeta != nullptr) P.fin_dbeta[c] += (float)P.red[c];
            if (P.fin_dgamma != nullptr) P.fin_dgamma[c] += (float)P.red[C + c];
            if (P.fin_dbias != nullptr && !P.training) P.fin_dbias[c] += __ldg(P.scale + c) * (float)P.red[c];
            if (c == 0 && P.fin_dslope != nullptr) P.fin_dslope[0] += (float)P.red[2 * C];
        }
        float mean[8], invstd[8];
        load_affine(P.mean, P.invstd, c8, mean, invstd);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (P.training) {
                const float m1 = (float)(P.red[c8 * 8 + i] * P.inv_count);
                const float m2 = (float)(P.red[C + c8 * 8 + i] * P.inv_count);
                ka[i] = -sc[i] * (m1 - m2 * mean[i] * invstd[i]);
                kb[i] = -sc[i] * m2 * invstd[i];
            } else {
                ka[i] = 0.0f; kb[i] = 0.0f;
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) { ka[i] = 0.0f; kb[i] = 0.0f; }
    }
    const int chunks = (HW + kBwdV * kThreads - 1) / (kBwdV * kThreads);
    const int items = P.N * P.D * chunks;
    const int W2 = P.W >> 1, HW2 = (P.H >> 1) * W2;
    // (nd, ch) = divmod(item, chunks) and the plane base pointers are stepped, not recomputed (no division and no
    // 64-bit multiply chains in the loop)
    const int step_nd = gridDim.x / chunks, step_ch = gridDim.x - step_nd * chunks;
    int nd = blockIdx.x / chunks, ch = blockIdx.x - nd * chunks;
    const int64_t y_stride = (int64_t)P.C8 * HW, g_stride = (int64_t)P.g1_c8tot * HW;
    const bf16x8* yp = P.y + ((int64_t)nd * P.C8 + c8) * HW + threadIdx.x;
    const bf16x8* g1p = P.g1 != nullptr ? P.g1 + ((int64_t)nd * P.g1_c8tot + P.g1_c8off + c8) * HW + threadIdx.x : nullptr;
    const int64_t dy_off = APPLY ? reinterpret_cast<const char*>(P.dy) - reinterpret_cast<const char*>(P.y) : 0;
    int pn = 0, pd = 0;          // POOL: (n, d) of plane nd
    if (POOL) { pn = nd / P.D; pd = nd - pn * P.D; }
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const bf16x8* gpp = nullptr;
        const uint2* idxp = nullptr;
        uint32_t code_d = 0;
        if (POOL) {
            const int kd = P.pool_kd;
            const int d2 = kd == 2 ? pd >> 1 : pd;
            const int64_t pnd = (int64_t)pn * (kd == 2 ? P.D >> 1 : P.D) + d2;
            gpp = P.g_pool + (pnd * P.gp_c8tot + P.gp_c8off + c8) * HW2;
            idxp = P.pool_idx + (pnd * P.C8 + c8) * HW2;
            code_d = (uint32_t)(pd - d2 * kd) * 4u;
        }
        const int voff = ch * (kBwdV * kThreads);
        int hwk[kBwdV];
        bool act[kBwdV];
#pragma unroll
        for (int k = 0; k < kBwdV; ++k) { hwk[k] = voff + (int)threadIdx.x + k * kThreads; act[k] = hwk[k] < HW; }
        int4 ry[kBwdV], rg[kBwdV], rp[kBwdV];
        uint2 rc[kBwdV];
        uint32_t mycode[kBwdV];
#pragma unroll
        for (int k = 0; k < kBwdV; ++k) {
            ry[k] = rg[k] = rp[k] = make_int4(0, 0, 0, 0);
            rc[k] = make_uint2(0, 0);
            mycode[k] = 0xffu;
            if (act[k]) {
                ry[k] = ld_stream16(yp + voff + k * kThreads);
                if (g1p != nullptr) rg[k] = ld_stream16(g1p + voff + k * kThreads);
                if (POOL) {
                    const int h = P.w_shift >= 0 ? hwk[k] >> P.w_shift : hwk[k] / P.W;
                    const int w = hwk[k] - h * P.W;
                    const int pix = (h >> 1) * W2 + (w >> 1);
                    mycode[k] = code_d + (uint32_t)((h & 1) * 2 + (w & 1));
                    rc[k] = __ldg(idxp + pix);
                    rp[k] = __ldg(reinterpret_cast<const int4*>(gpp + pix));
                }
            }
        }
#pragma unroll
        for (int k = 0; k < kBwdV; ++k) {
            if (!act[k]) continue;
            float yf[8], g[8];
            bf16x8_to_float(*reinterpret_cast<bf16x8*>(&ry[k]), yf);
            bf16x8_to_float(*reinterpret_cast<bf16x8*>(&rg[k]), g);
            if (POOL) {
                // byte-wise compare of the 8 argmax codes with this voxel's code, widened to bf16 masks: the pooled
                // gradient is masked in its packed form (2 + 4 + 4 integer ops for 8 channels)
                const uint32_t code4 = mycode[k] * 0x01010101u;
                const uint32_t m0 = __vcmpeq4(rc[k].x, code4), m1 = __vcmpeq4(rc[k].y, code4);
                rp[k].x &= (int)__byte_perm(m0, 0, 0x1100); rp[k].y &= (int)__byte_perm(m0, 0, 0x3322);
                rp[k].z &= (int)__byte_perm(m1, 0, 0x1100); rp[k].w &= (int)__byte_perm(m1, 0, 0x3322);
                float gp[8];
                bf16x8_to_float(*reinterpret_cast<bf16x8*>(&rp[k]), gp);
#pragma unroll
                for (int i = 0; i < 8; ++i) g[i] += gp[i];
            }
            if (DROP) {
                const uint32_t keep = keep_bits(P.drop_mask, seed, P.offset, (yp - P.y) + (hwk[k] - (int)threadIdx.x), P.drop_p);
#pragma unroll
                for (int i = 0; i < 8; ++i) g[i] = ((keep >> i) & 1u) ? g[i] * keep_scale : 0.0f;
            }
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float z = fmaf(yf[i], sc[i], sh[i]);
                const bool pos = z > 0.0f;
                const float dz = pos ? g[i] : g[i] * slope;
                if (!APPLY) {
                    dsl = fmaf(z, pos ? 0.0f : g[i], dsl);
                    ka[i] += dz;
                    kb[i] = fmaf(dz, yf[i], kb[i]);
                } else {
                    o[i] = fmaf(sc[i], dz, fmaf(kb[i], yf[i], ka[i]));
                }
            }
            if (APPLY)
                st_bf16x8(const_cast<char*>(reinterpret_cast<const char*>(yp + voff + k * kThreads)) + dy_off, o);
        }
        // next item
        int dnd = step_nd;
        ch += step_ch;
        if (ch >= chunks) { ch -= chunks; ++dnd; }
        yp += dnd * y_stride;
        if (g1p != nullptr) g1p += dnd * g_stride;
        if (POOL) {
            pd += dnd;
            while (pd >= P.D) { pd -= P.D; ++pn; }
        }
    }
    FPL_PDL_TRIGGER();       // main loop done: the next kernel of the stream may be scheduled as blocks drain
    if (!APPLY) {
        __shared__ float sm[kThreads / 32][17];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float a = warp_sum(ka[i]), b = warp_sum(kb[i]);
            if (lane == 0) { sm[wid][i] = a; sm[wid][8 + i] = b; }
        }
        float c = warp_sum(dsl);
        if (lane == 0) sm[wid][16] = c;
        __syncthreads();
        if (threadIdx.x < 17) {
            float t = 0.0f;
#pragma unroll
            for (int k = 0; k < kThreads / 32; ++k) t += sm[k][threadIdx.x];
            const int i = threadIdx.x;
            if (i < 8) {
                atomicAdd(P.red + c8 * 8 + i, (double)t);
            } else if (i < 16) {
                // sum dz*xhat = invstd * (sum dz*y - mean * sum dz)
                float t1 = 0.0f;
#pragma unroll
                for (int k = 0; k < kThreads / 32; ++k) t1 += sm[k][i - 8];
                const int c = c8 * 8 + (i - 8);
                const double v = (double)__ldg(P.invstd + c) * ((double)t - (double)__ldg(P.mean + c) * (double)t1);
                atomicAdd(P.red + C + c, v);
            } else {
                atomicAdd(P.red + 2 * C, (double)t);
            }
        }
    }
}

__global__ void dsbn_bwd_finalize_kernel(const double* __restrict__ red, const float* __restrict__ scale, int training,
                                         float* dgamma, float* dbeta, float* dslope, float* dbias_conv,
                                         const float* __restrict__ invstd, int C) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < C) {
        // dz is the gradient wrt the BN output: dbeta = sum dz, dgamma = sum dz*xhat
        if (dbeta != nullptr) dbeta[c] += (float)red[c];
        if (dgamma != nullptr) dgamma[c] += (float)red[C + c];
        // the conv bias feeds straight into BN: in training mode its gradient is identically 0
        // (sum_v dy = 0), in eval mode it is scale * sum dz
        if (dbias_conv != nullptr && !training) dbias_conv[c] += scale[c] * (float)red[c];
    }
    if (c == 0 && dslope != nullptr) dslope[0] += (float)red[2 * C];
}

}  // namespace

constexpr int g_bwd_blocks_per_sm = 8;

extern "C" int fpl_dsbn_finalize(const double* stats, int64_t count, const float* gamma, const float* beta,
                                 float* running_mean, float* running_var, int64_t* num_batches_tracked,
                                 float momentum, float eps, int training, float* scale, float* shift,
                                 float* save_mean, float* save_invstd, int c, void* stream) {
    FPL_REQUIRE(c > 0 && c % 8 == 0, "fpl_dsbn_finalize: channels (%d) must be a positive multiple of 8", c);
    FPL_REQUIRE(training ? (stats != nullptr && count > 0) : (running_mean != nullptr && running_var != nullptr),
                "fpl_dsbn_finalize: missing statistics for training=%d", training);
    double unbias = count > 1 ? (double)count / (double)(count - 1) : 1.0;
    fpl_launch(dsbn_finalize_kernel, (c + 127) / 128, 128, 0, (cudaStream_t)stream, 
        stats, 1.0 / (double)(count > 0 ? count : 1), unbias, gamma, beta, running_mean, running_var,
        (long long*)num_batches_tracked, momentum, eps, training, scale, shift, save_mean, save_invstd, c);
    FPL_LAUNCH_CHECK();
    return 0;
}

static int act_fwd_launch(const BnFinalize* fin, const void* y, const float* scale, const float* shift, const float* slope,
                                void* a, int a_c8tot, int a_c8off, void* pooled, int p_c8tot, int p_c8off,
                                uint8_t* pool_idx, int pool_kd, float drop_p, const uint8_t* drop_mask,
                                uint64_t seed, uint64_t offset, const uint64_t* seed_dev, int n, int d, int h, int w, int c,
                                void* stream) {
    FPL_REQUIRE(c > 0 && c % 8 == 0, "fpl_dsbn_act_fwd: channels (%d) must be a multiple of 8", c);
    FPL_REQUIRE(drop_p >= 0.0f && drop_p < 1.0f, "fpl_dsbn_act_fwd: dropout p=%f out of [0,1)", drop_p);
    ActParams P;
    if (fin != nullptr) { P.fin = *fin; P.fin.enabled = 1; } else P.fin.enabled = 0;
    P.y = (const bf16x8*)y; P.scale = scale; P.shift = shift; P.slope = slope;
    P.a = (bf16x8*)a; P.a_c8tot = a_c8tot; P.a_c8off = a_c8off;
    P.pooled = (bf16x8*)pooled; P.p_c8tot = p_c8tot; P.p_c8off = p_c8off; P.pool_idx = (uint2*)pool_idx;
    P.pool_kd = pool_kd; P.drop_p = drop_p; P.drop_mask = (const uint2*)drop_mask; P.seed = seed; P.offset = offset;
    P.seed_dev = (const unsigned long long*)seed_dev;
    P.N = n; P.D = d; P.C8 = c / 8; P.H = h; P.W = w;
    const int c8 = c / 8;
    if (pooled != nullptr) {
        FPL_REQUIRE(pool_kd == 1 || pool_kd == 2, "fpl_dsbn_act_fwd: pool_kd must be 1 or 2");
        FPL_REQUIRE(h % 2 == 0 && w % 2 == 0 && d % pool_kd == 0, "fpl_dsbn_act_fwd: pooled dims must be even");
        FPL_REQUIRE(drop_p == 0.0f, "fpl_dsbn_act_fwd: dropout is not combined with pooling");
        FPL_REQUIRE(pool_idx != nullptr, "fpl_dsbn_act_fwd: pool_idx required");
        const int64_t hw2 = (int64_t)(h / 2) * (w / 2);
        const int64_t items = (int64_t)n * (d / pool_kd) * ((hw2 + kThreads - 1) / kThreads);
        int64_t bx = (FPL_NUM_SMS * 8 + c8 - 1) / c8;
        if (bx > items) bx = items;
        if (bx < 1) bx = 1;
        fpl_launch(dsbn_act_pool_fwd_kernel, dim3((unsigned)bx, (unsigned)c8), kThreads, 0, (cudaStream_t)stream, P);
    } else {
        const int64_t hw = (int64_t)h * w;
        const int64_t items = (int64_t)n * d * ((hw + 2 * kThreads - 1) / (2 * kThreads));
        int64_t bx = (FPL_NUM_SMS * 8 + c8 - 1) / c8;
        if (bx > items) bx = items;
        if (bx < 1) bx = 1;
        fpl_launch(dsbn_act_fwd_kernel, dim3((unsigned)bx, (unsigned)c8), kThreads, 0, (cudaStream_t)stream, P);
    }
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_dsbn_act_fwd(const void* y, const float* scale, const float* shift, const float* slope,
                                void* a, int a_c8tot, int a_c8off, void* pooled, int p_c8tot, int p_c8off,
                                uint8_t* pool_idx, int pool_kd, float drop_p, const uint8_t* drop_mask,
                                uint64_t seed, uint64_t offset, const uint64_t* seed_dev, int n, int d, int h, int w, int c,
                                void* stream) {
    return act_fwd_launch(nullptr, y, scale, shift, slope, a, a_c8tot, a_c8off, pooled, p_c8tot, p_c8off, pool_idx, pool_kd,
                          drop_p, drop_mask, seed, offset, seed_dev, n, d, h, w, c, stream);
}

extern "C" int fpl_dsbn_bn_act_fwd(const void* y, const double* stats, int64_t count, const float* gamma, const float* beta,
                                   float* running_mean, float* running_var, int64_t* num_batches_tracked, float momentum,
                                   float eps, int training, float* scale, float* shift, float* save_mean,
                                   float* save_invstd, const float* slope, void* a, int a_c8tot, int a_c8off, void* pooled,
                                   int p_c8tot, int p_c8off, uint8_t* pool_idx, int pool_kd, float drop_p,
                                   const uint8_t* drop_mask, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                                   int n, int d, int h, int w, int c, void* stream) {
    FPL_REQUIRE(training ? (stats != nullptr && count > 0) : (running_mean != nullptr && running_var != nullptr),
                "fpl_dsbn_bn_act_fwd: missing statistics for training=%d", training);
    FPL_REQUIRE(scale && shift && save_mean && save_invstd && gamma && beta, "fpl_dsbn_bn_act_fwd: NULL parameter arrays");
    BnFinalize F;
    F.stats = stats; F.inv_count = 1.0 / (double)(count > 0 ? count : 1);
    F.unbias = count > 1 ? (double)count / (double)(count - 1) : 1.0;
    F.gamma = gamma; F.beta = beta; F.running_mean = running_mean; F.running_var = running_var;
    F.nbt = (long long*)num_batches_tracked; F.momentum = momentum; F.eps = eps; F.training = training; F.enabled = 1;
    F.scale = scale; F.shift = shift; F.save_mean = save_mean; F.save_invstd = save_invstd;
    return act_fwd_launch(&F, y, scale, shift, slope, a, a_c8tot, a_c8off, pooled, p_c8tot, p_c8off, pool_idx, pool_kd,
                          drop_p, drop_mask, seed, offset, seed_dev, n, d, h, w, c, stream);
}

static int fill_bwd(ActBwdParams& P, const void* y, const void* g1, int g1_c8tot, int g1_c8off, const void* g_pool,
                    int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd, const float* scale,
                    const float* shift, const float* save_mean, const float* save_invstd, const float* slope,
                    float drop_p, const uint8_t* drop_mask, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                    int n, int d, int h, int w, int c) {
    FPL_REQUIRE(c > 0 && c % 8 == 0, "dsbn bwd: channels (%d) must be a multiple of 8", c);
    FPL_REQUIRE(g1 != nullptr || g_pool != nullptr, "dsbn bwd: no incoming gradient");
    if (g_pool != nullptr) {
        FPL_REQUIRE(pool_idx != nullptr && (pool_kd == 1 || pool_kd == 2), "dsbn bwd: pool_idx/pool_kd invalid");
        FPL_REQUIRE(h % 2 == 0 && w % 2 == 0 && d % pool_kd == 0, "dsbn bwd: pooled dims must be even");
    }
    P.y = (const bf16x8*)y; P.g1 = (const bf16x8*)g1; P.g1_c8tot = g1_c8tot; P.g1_c8off = g1_c8off;
    P.g_pool = (const bf16x8*)g_pool; P.gp_c8tot = gp_c8tot; P.gp_c8off = gp_c8off;
    P.pool_idx = (const uint2*)pool_idx; P.pool_kd = pool_kd > 0 ? pool_kd : 2;
    P.scale = scale; P.shift = shift; P.mean = save_mean; P.invstd = save_invstd; P.slope = slope;
    P.drop_p = drop_p; P.drop_mask = (const uint2*)drop_mask; P.seed = seed; P.offset = offset;
    P.seed_dev = (const unsigned long long*)seed_dev;
    P.red = nullptr; P.dy = nullptr; P.training = 1;
    P.fin_dgamma = P.fin_dbeta = P.fin_dslope = P.fin_dbias = nullptr; P.inv_count = 1.0 / ((double)n * d * h * w);
    P.N = n; P.D = d; P.C8 = c / 8; P.H = h; P.W = w;
    P.w_shift = -1;
    for (int s = 0; s < 16; ++s) if ((1 << s) == w) P.w_shift = s;
    return 0;
}

// blocks per channel group: enough blocks for ~8 per SM over the whole grid, at most one per work item
static dim3 bwd_grid(int n, int d, int h, int w, int c) {
    const int64_t hw = (int64_t)h * w;
    const int64_t chunks = (hw + kBwdV * kThreads - 1) / (kBwdV * kThreads);
    const int64_t items = (int64_t)n * d * chunks;
    const int c8 = c / 8;
    int64_t bx = (FPL_NUM_SMS * g_bwd_blocks_per_sm + c8 - 1) / c8;
    if (bx > items) bx = items;
    if (bx < 1) bx = 1;
    return dim3((unsigned)bx, (unsigned)c8);
}

template <bool APPLY>
static void bwd_dispatch(const ActBwdParams& P, dim3 grid, cudaStream_t stream) {
    const bool pool = P.g_pool != nullptr, drop = P.drop_p > 0.0f;
    if (pool && drop) fpl_launch(dsbn_act_bwd_kernel<APPLY, true, true>, grid, kThreads, 0, stream, P);
    else if (pool) fpl_launch(dsbn_act_bwd_kernel<APPLY, true, false>, grid, kThreads, 0, stream, P);
    else if (drop) fpl_launch(dsbn_act_bwd_kernel<APPLY, false, true>, grid, kThreads, 0, stream, P);
    else fpl_launch(dsbn_act_bwd_kernel<APPLY, false, false>, grid, kThreads, 0, stream, P);
}

extern "C" int fpl_dsbn_act_bwd_reduce(const void* y, const void* g1, int g1_c8tot, int g1_c8off, const void* g_pool,
                                       int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                                       const float* scale, const float* shift, const float* save_mean,
                                       const float* save_invstd, const float* slope, float drop_p,
                                       const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                                       const uint64_t* seed_dev, double* red, int n, int d, int h, int w, int c,
                                       void* stream) {
    ActBwdParams P;
    int rc = fill_bwd(P, y, g1, g1_c8tot, g1_c8off, g_pool, gp_c8tot, gp_c8off, pool_idx, pool_kd, scale, shift,
                      save_mean, save_invstd, slope, drop_p, drop_mask, seed, offset, seed_dev, n, d, h, w, c);
    if (rc) return rc;
    P.red = red;
    bwd_dispatch<false>(P, bwd_grid(n, d, h, w, c), (cudaStream_t)stream);
    FPL_LAUNCH_CHECK();
    return 0;
}

static int act_bwd_apply_launch(float* dgamma, float* dbeta, float* dslope, float* dbias_conv, const void* y, const void* g1, int g1_c8tot, int g1_c8off, const void* g_pool,
                                      int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                                      const float* scale, const float* shift, const float* save_mean,
                                      const float* save_invstd, const float* slope, float drop_p,
                                      const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                                      const uint64_t* seed_dev, const double* red, int training, void* dy, int n, int d,
                                      int h, int w, int c, void* stream) {
    ActBwdParams P;
    int rc = fill_bwd(P, y, g1, g1_c8tot, g1_c8off, g_pool, gp_c8tot, gp_c8off, pool_idx, pool_kd, scale, shift,
                      save_mean, save_invstd, slope, drop_p, drop_mask, seed, offset, seed_dev, n, d, h, w, c);
    if (rc) return rc;
    P.red = const_cast<double*>(red);
    P.dy = (bf16x8*)dy;
    P.training = training;
    P.fin_dgamma = dgamma; P.fin_dbeta = dbeta; P.fin_dslope = dslope; P.fin_dbias = dbias_conv;
    bwd_dispatch<true>(P, bwd_grid(n, d, h, w, c), (cudaStream_t)stream);
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_dsbn_act_bwd_apply(const void* y, const void* g1, int g1_c8tot, int g1_c8off, const void* g_pool,
                                      int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                                      const float* scale, const float* shift, const float* save_mean,
                                      const float* save_invstd, const float* slope, float drop_p,
                                      const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                                      const uint64_t* seed_dev, const double* red, int training, void* dy, int n, int d,
                                      int h, int w, int c, void* stream) {
    return act_bwd_apply_launch(nullptr, nullptr, nullptr, nullptr, y, g1, g1_c8tot, g1_c8off, g_pool, gp_c8tot, gp_c8off, pool_idx, pool_kd, scale, shift, save_mean, save_invstd, slope, drop_p, drop_mask, seed, offset, seed_dev, red, training, dy, n, d, h, w, c, stream);
}

extern "C" int fpl_dsbn_act_bwd_apply_fin(const void* y, const void* g1, int g1_c8tot, int g1_c8off, const void* g_pool,
                                      int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                                      const float* scale, const float* shift, const float* save_mean,
                                      const float* save_invstd, const float* slope, float drop_p,
                                      const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                                      const uint64_t* seed_dev, const double* red, int training, void* dy, int n, int d,
                                      int h, int w, int c, void* stream, float* dgamma, float* dbeta, float* dslope, float* dbias_conv) {
    return act_bwd_apply_launch(dgamma, dbeta, dslope, dbias_conv, y, g1, g1_c8tot, g1_c8off, g_pool, gp_c8tot, gp_c8off, pool_idx, pool_kd, scale, shift, save_mean, save_invstd, slope, drop_p, drop_mask, seed, offset, seed_dev, red, training, dy, n, d, h, w, c, stream);
}

extern "C" int fpl_dsbn_bwd_finalize(const double* red, const float* scale, const float* save_invstd, int training,
                                     float* dgamma, float* dbeta, float* dslope, float* dbias_conv, int c,
                                     void* stream) {
    fpl_launch(dsbn_bwd_finalize_kernel, (c + 127) / 128, 128, 0, (cudaStream_t)stream, red, scale, training, dgamma, dbeta,
                                                                                dslope, dbias_conv, save_invstd, c);
    FPL_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------
// eval-mode affine maps of all conv units of a forward pass in ONE launch (inference epilogue of the conv kernels)
// ------------------------------------------------------------------------------------
namespace {
constexpr int kMaxAffine = 48;
struct AffineBatch {
    const float* gamma[kMaxAffine];
    const float* beta[kMaxAffine];
    const float* mean[kMaxAffine];
    const float* var[kMaxAffine];
    const float* bias[kMaxAffine];      // conv bias feeding the BatchNorm (may be NULL)
    float* scale[kMaxAffine];
    float* shift[kMaxAffine];
    int c[kMaxAffine];
    float eps;
};
__global__ void dsbn_eval_affine_batch_kernel(const __grid_constant__ AffineBatch B) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int e = blockIdx.y;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B.c[e]; i += gridDim.x * blockDim.x) {
        const float invstd = 1.0f / sqrtf(B.var[e][i] + B.eps);      // same expression as the eval branch of bn_prologue
        const float g = B.gamma[e][i] * invstd;
        const float b = B.bias[e] != nullptr ? B.bias[e][i] : 0.0f;
        B.scale[e][i] = g;
        B.shift[e][i] = (B.beta[e][i] - B.mean[e][i] * g) + b * g;
    }
}
}  // namespace

extern "C" int fpl_dsbn_eval_affine_batch(int count, const float* const* h_gamma, const float* const* h_beta,
                                          const float* const* h_running_mean, const float* const* h_running_var,
                                          const float* const* h_conv_bias, float* const* h_scale, float* const* h_shift,
                                          const int* h_c, float eps, void* stream) {
    FPL_REQUIRE(count >= 0 && count <= kMaxAffine, "fpl_dsbn_eval_affine_batch: count %d not in [0,%d]", count, kMaxAffine);
    if (count == 0) return 0;
    AffineBatch B;
    int cmax = 0;
    for (int e = 0; e < count; ++e) {
        FPL_REQUIRE(h_gamma[e] && h_beta[e] && h_running_mean[e] && h_running_var[e] && h_scale[e] && h_shift[e] && h_c[e] > 0,
                    "fpl_dsbn_eval_affine_batch: NULL array in entry %d", e);
        B.gamma[e] = h_gamma[e]; B.beta[e] = h_beta[e]; B.mean[e] = h_running_mean[e]; B.var[e] = h_running_var[e];
        B.bias[e] = h_conv_bias != nullptr ? h_conv_bias[e] : nullptr; B.scale[e] = h_scale[e]; B.shift[e] = h_shift[e];
        B.c[e] = h_c[e];
        if (h_c[e] > cmax) cmax = h_c[e];
    }
    B.eps = eps;
    fpl_launch(dsbn_eval_affine_batch_kernel, dim3((cmax + 127) / 128, count), 128, 0, (cudaStream_t)stream, B);
    FPL_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------
// max-pool only (inference: the activation was already written by the conv epilogue)
// ------------------------------------------------------------------------------------
namespace {
struct PoolParams {
    const bf16x8* a;
    int a_c8tot, a_c8off;
    bf16x8* pooled;
    int p_c8tot, p_c8off;
    int kd, N, D, C8, H, W;
};
// grid: (chunks of H2*W2, N*D2*C8 pooled planes); one thread per pooled vector
__global__ void __launch_bounds__(kThreads) maxpool_c8_kernel(PoolParams P) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int kd = P.kd, D2 = P.D / kd, H2 = P.H / 2, W2 = P.W / 2;
    const int HW = P.H * P.W, HW2 = H2 * W2;
    const int pplane = blockIdx.y;
    const int c8 = pplane % P.C8;
    const int nd2 = pplane / P.C8;
    const int d2 = nd2 % D2, n = nd2 / D2;
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < HW2; v += gridDim.x * blockDim.x) {
        const int h2 = v / W2, w2 = v - h2 * W2;
        int4 raw[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int dd = q >> 2, hh = (q >> 1) & 1, ww = q & 1;
            if (dd < kd) {
                const int64_t nd = (int64_t)n * P.D + d2 * kd + dd;
                raw[q] = ld_stream16(P.a + (nd * P.a_c8tot + P.a_c8off + c8) * HW + (h2 * 2 + hh) * P.W + w2 * 2 + ww);
            }
        }
        float best[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) best[i] = -INFINITY;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if ((q >> 2) < kd) {
                float f[8];
                bf16x8_to_float(*reinterpret_cast<bf16x8*>(&raw[q]), f);
#pragma unroll
                for (int i = 0; i < 8; ++i) best[i] = fmaxf(best[i], f[i]);
            }
        }
        st_bf16x8(P.pooled + ((int64_t)nd2 * P.p_c8tot + P.p_c8off + c8) * HW2 + v, best);
    }
}
}  // namespace

extern "C" int fpl_maxpool_c8(const void* a, int a_c8tot, int a_c8off, void* pooled, int p_c8tot, int p_c8off, int pool_kd,
                              int n, int d, int h, int w, int c, void* stream) {
    FPL_REQUIRE(c > 0 && c % 8 == 0, "fpl_maxpool_c8: channels (%d) must be a multiple of 8", c);
    FPL_REQUIRE(pool_kd == 1 || pool_kd == 2, "fpl_maxpool_c8: pool_kd must be 1 or 2");
    FPL_REQUIRE(h % 2 == 0 && w % 2 == 0 && d % pool_kd == 0, "fpl_maxpool_c8: pooled dims must be even");
    FPL_REQUIRE(a != nullptr && pooled != nullptr, "fpl_maxpool_c8: NULL buffer");
    PoolParams P;
    P.a = (const bf16x8*)a; P.a_c8tot = a_c8tot; P.a_c8off = a_c8off; P.pooled = (bf16x8*)pooled; P.p_c8tot = p_c8tot;
    P.p_c8off = p_c8off; P.kd = pool_kd; P.N = n; P.D = d; P.C8 = c / 8; P.H = h; P.W = w;
    const int64_t planes = (int64_t)n * (d / pool_kd) * (c / 8);
    FPL_REQUIRE(planes <= 65535, "fpl_maxpool_c8: too many planes (%lld)", (long long)planes);
    const int hw2 = (h / 2) * (w / 2);
    fpl_launch(maxpool_c8_kernel, dim3((hw2 + kThreads - 1) / kThreads, (unsigned)planes), kThreads, 0, (cudaStream_t)stream, P);
    FPL_LAUNCH_CHECK();
    return 0;
}

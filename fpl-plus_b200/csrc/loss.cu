// Fused pixel/image-weighted Dice + cross-entropy: reduction pass and gradient pass.
// Replaces DiceLoss (PyMIC/pymic/loss/seg/dice.py:20-57), get_classwise_dice
// (loss/seg/util.py:85-107), CrossEntropyLoss (loss/seg/ce.py:23-44), CombinedLoss
// (loss/seg/combined.py:34-39) and the training-time hard-Dice metric
// (net_run_dsbn/agent_seg.py:472-476).  Pure HBM streaming over NCDHW fp32 (the layout the
// PyMIC loss API hands over): 8C+4 bytes/voxel in the reduce pass, 12C+4 in the grad pass.
#include <cstdlib>
#include "common.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kThreads = 256;

template <int C>
__device__ __forceinline__ void softmax_c(const float* z, float* p) {
    if (C == 2) {
        // exp(z_max - z_max) is exactly 1: one expf instead of two, same bits as the general form below
        const bool first = z[0] >= z[1];
        const float e = expf(first ? z[1] - z[0] : z[0] - z[1]);
        const float inv = 1.0f / (1.0f + e);
        p[0] = first ? inv : e * inv;
        p[1] = first ? e * inv : inv;
        return;
    }
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float s = 0.0f;
#pragma unroll
    for (int c = 0; c < C; ++c) { p[c] = expf(z[c] - m); s += p[c]; }
    float inv = 1.0f / s;
#pragma unroll
    for (int c = 0; c < C; ++c) p[c] *= inv;
}

// Where the ground truth and the pixel weight of a voxel come from.  The PyMIC loss API hands fp32 one-hot / soft labels
// [N,C,D,H,W] and an fp32 weight map [N,1,D,H,W]; the device data path (SURVEY 8 f-3) hands a uint8 label map [N,D,H,W]
// (one-hot built here: LabelToProbability, transform/label_convert.py:82-88) and a uint8 agreement code [N,D,H,W]
// (0, 1, 2 = weight 0, 0.5, 1 of data/get_pixel_weight.py:21-26) with the per-sample image weight folded in here
// exactly as NiftyDataset.set_weight_ does (io/nifty_dataset.py:165-168: w < 1 -> 0, else w * image_weight).
struct LossSrc {
    const float* soft_y;      // fp32 [N,C,S] or NULL
    const uint8_t* label;     // u8 [N,S] (used when soft_y == NULL)
    const float* weight;      // fp32 [N,S] or NULL
    const uint8_t* wcode;     // u8 [N,S] or NULL (used when weight == NULL)
    const float* image_w;     // fp32 [N] or NULL: fold the image weight into wcode (set_weight_)
    int prob_input;           // loss_softmax = False (loss/seg/abstract.py:16-21): `logits` already are probabilities
};

// One float4 group (4 voxels) of inputs as it comes from memory.  Loading and decoding are separate so that a thread can
// issue the loads of U groups back to back (one DRAM round trip per batch) before the first use stalls it.
template <int C, bool LEAN>
struct RawGroup {
    float4 z[C];
    float4 y[C];              // soft_y layout
    float4 wf;                // fp32 weight layout
    uint32_t lab, code;       // uint8 layouts
};
template <int C>
struct RawGroup<C, true> {    // uint8 labels, uint8 weight codes or no weights: 4C + 2 registers per group
    float4 z[C];
    uint32_t lab, code;
};

template <int C, bool LEAN>
__device__ __forceinline__ void load_raw(const float* __restrict__ logits, const LossSrc& src, int64_t n, int64_t s4, int64_t S4,
                                         RawGroup<C, LEAN>& r) {
#pragma unroll
    for (int c = 0; c < C; ++c) r.z[c] = ld_stream_f4(reinterpret_cast<const float4*>(logits) + (n * C + c) * S4 + s4);
    if constexpr (!LEAN) {
        if (src.soft_y != nullptr) {
#pragma unroll
            for (int c = 0; c < C; ++c) r.y[c] = ld_stream_f4(reinterpret_cast<const float4*>(src.soft_y) + (n * C + c) * S4 + s4);
        }
        if (src.weight != nullptr) r.wf = ld_stream_f4(reinterpret_cast<const float4*>(src.weight) + n * S4 + s4);
    }
    if (LEAN || src.soft_y == nullptr) r.lab = __ldg(reinterpret_cast<const uint32_t*>(src.label) + n * S4 + s4);
    if ((LEAN || src.weight == nullptr) && src.wcode != nullptr) r.code = __ldg(reinterpret_cast<const uint32_t*>(src.wcode) + n * S4 + s4);
}

template <int C, bool LEAN>
__device__ __forceinline__ void decode_truth4(const LossSrc& src, const RawGroup<C, LEAN>& r, float4 (&yv)[C]) {
    bool soft = false;
    if constexpr (!LEAN) {
        soft = src.soft_y != nullptr;
        if (soft) {
#pragma unroll
            for (int c = 0; c < C; ++c) yv[c] = r.y[c];
        }
    }
    if (!soft) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int l = (int)((r.lab >> (8 * j)) & 0xffu);
#pragma unroll
            for (int c = 0; c < C; ++c) reinterpret_cast<float*>(&yv[c])[j] = (l == c) ? 1.0f : 0.0f;
        }
    }
}

template <int C, bool LEAN>
__device__ __forceinline__ float4 decode_weight4(const LossSrc& src, const RawGroup<C, LEAN>& r, float iw) {
    if constexpr (!LEAN) {
        if (src.weight != nullptr) return r.wf;
    }
    if (src.wcode == nullptr) return make_float4(1.f, 1.f, 1.f, 1.f);
    const bool fold = src.image_w != nullptr;
    float4 w;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float a = 0.5f * (float)((r.code >> (8 * j)) & 0xffu);
        reinterpret_cast<float*>(&w)[j] = fold ? (a < 1.0f ? 0.0f : a) * iw : a;
    }
    return w;
}

// sums layout (double): I[C], Y[C], P[C], sum_w, sum_w_ce, HI[C], HY[C], HP[C], sum_c,v p*log2(p + 1e-10)
// grid = (blocks per sample, N): the sample index is blockIdx.y (no 64-bit division per group); a thread walks its groups
// in batches of U whose loads are all issued before the first is used.
template <int C, int U, bool LEAN>
__global__ void __launch_bounds__(kThreads, LEAN ? (C == 2 ? (U == 8 ? 2 : (U == 2 ? 4 : 3)) : (C <= 3 ? 3 : 2)) : 1) dice_ce_reduce_kernel(const float* __restrict__ logits, LossSrc src,
                                                                 double* sums, int N, int64_t S4, int want_entropy) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const bool weighted = src.weight != nullptr || src.wcode != nullptr;
    constexpr int NV = 6 * C + 3;
    float acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = 0.0f;
    const int64_t n = blockIdx.y;
    const float iw = src.image_w != nullptr && src.wcode != nullptr && src.weight == nullptr ? __ldg(src.image_w + n) : 1.0f;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g0 < S4; g0 += U * stride) {
        RawGroup<C, LEAN> raw[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (g0 + u * stride < S4) load_raw<C, LEAN>(logits, src, n, g0 + u * stride, S4, raw[u]);
#pragma unroll
        for (int u = 0; u < U; ++u) {
        if (g0 + u * stride >= S4) break;
        float4 yv[C];
        decode_truth4<C, LEAN>(src, raw[u], yv);
        float4 wv = make_float4(1.f, 1.f, 1.f, 1.f);
        if (weighted) wv = decode_weight4<C, LEAN>(src, raw[u], iw);
        const float4 (&zv)[C] = raw[u].z;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float z[C], y[C], p[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                z[c] = reinterpret_cast<const float*>(&zv[c])[j];
                y[c] = reinterpret_cast<const float*>(&yv[c])[j];
            }
            float w = reinterpret_cast<const float*>(&wv)[j];
            if (src.prob_input) {
#pragma unroll
                for (int c = 0; c < C; ++c) p[c] = z[c];
            } else {
                softmax_c<C>(z, p);
            }
            if (want_entropy) {
#pragma unroll
                for (int c = 0; c < C; ++c) acc[6 * C + 2] = fmaf(p[c], log2f(p[c] + 1e-10f), acc[6 * C + 2]);
            }
            int am = 0;
            float best = z[0];
            float ce = 0.0f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                if (c > 0 && z[c] > best) { best = z[c]; am = c; }
                acc[c] = fmaf(w * y[c], p[c], acc[c]);
                acc[C + c] = fmaf(w, y[c], acc[C + c]);
                acc[2 * C + c] = fmaf(w, p[c], acc[2 * C + c]);
                if (y[c] != 0.0f) ce -= y[c] * logf(p[c] * 0.999f + 5e-4f);     // one-hot labels: one logf per voxel
                acc[3 * C + 2 + C + c] += y[c];
            }
            acc[3 * C] += w;
            acc[3 * C + 1] = fmaf(w, ce, acc[3 * C + 1]);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                if (c == am) {
                    acc[3 * C + 2 + c] += y[c];
                    acc[3 * C + 2 + 2 * C + c] += 1.0f;
                }
            }
        }
        }
    }
    __shared__ float sm[kThreads / 32][NV];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        float t = warp_sum(acc[i]);
        if (lane == 0) sm[wid][i] = t;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < kThreads / 32; ++k) t += (double)sm[k][threadIdx.x];
        atomicAdd(sums + threadIdx.x, t);
    }
}

template <int C, int U, bool LEAN>
__global__ void __launch_bounds__(kThreads, LEAN ? (C == 2 ? (U == 8 ? 2 : (U == 2 ? 4 : 3)) : (C <= 3 ? 3 : 2)) : 1) dice_ce_grad_kernel(const float* __restrict__ logits, LossSrc src,
                                                               const double* __restrict__ sums, float w_dice,
                                                               float w_ce, float w_ent, float grad_scale,
                                                               const float* __restrict__ grad_scale_dev, float* loss,
                                                               float* dlogits, int N, int64_t S4, int n_global,
                                                               double* hard_dice) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const bool weighted = src.weight != nullptr || src.wcode != nullptr;
    if (grad_scale_dev != nullptr) grad_scale *= __ldg(grad_scale_dev);
    // per-class constants of dDice/dp:  g_c = -(1/C) * w * (2*y*den - num) / den^2
    float a_c[C], b_c[C];
    double dice_mean = 0.0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        double I = sums[c], Y = sums[C + c], Pp = sums[2 * C + c];
        double den = Y + Pp + 1e-5, num = 2.0 * I + 1e-5;
        dice_mean += num / den;
        a_c[c] = (float)(-(double)w_dice * 2.0 / (C * den));          // * w * y
        b_c[c] = (float)((double)w_dice * num / (C * den * den));     // * w
    }
    dice_mean /= C;
    const double sum_w = sums[3 * C], sum_wce = sums[3 * C + 1];
    // voxels the sums cover: the local batch, or the GLOBAL batch when the sums were all-reduced (exact data-parallel mode)
    const double V = (double)(n_global > 0 ? n_global : N) * (double)S4 * 4.0;
    const double ce_den = weighted ? sum_w + 1e-5 : V;
    if (loss != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
        double l = 0.0;
        if (w_dice != 0.0f) l += (double)w_dice * (1.0 - dice_mean);
        if (w_ce != 0.0f) l += (double)w_ce * (sum_wce / ce_den);
        // entropy regulariser of agent_seg.py:353,467: -sum p*log2(p + 1e-10) / (N*D*H*W)
        if (w_ent != 0.0f) l += (double)w_ent * (-sums[6 * C + 2] / V);
        loss[0] = (float)l;
        // class-wise Dice of the argmax one-hot against the ground truth (agent_seg.py:472-476) from the hard counters
        if (hard_dice != nullptr) {
#pragma unroll
            for (int c = 0; c < C; ++c)
                hard_dice[c] = (2.0 * sums[3 * C + 2 + c] + 1e-5) / (sums[3 * C + 2 + C + c] + sums[3 * C + 2 + 2 * C + c] + 1e-5);
        }
    }
    if (dlogits == nullptr) return;
    const float ce_k = (float)(-(double)w_ce * 0.999 / ce_den);
    const float ent_k = (float)(-(double)w_ent / V);
    const int64_t n = blockIdx.y;
    const float iw = src.image_w != nullptr && src.wcode != nullptr && src.weight == nullptr ? __ldg(src.image_w + n) : 1.0f;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g0 < S4; g0 += U * stride) {
        RawGroup<C, LEAN> raw[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (g0 + u * stride < S4) load_raw<C, LEAN>(logits, src, n, g0 + u * stride, S4, raw[u]);
#pragma unroll
        for (int u = 0; u < U; ++u) {
        const int64_t s4 = g0 + u * stride;
        if (s4 >= S4) break;
        float4 yv[C], ov[C];
        decode_truth4<C, LEAN>(src, raw[u], yv);
        float4 wv = make_float4(1.f, 1.f, 1.f, 1.f);
        if (weighted) wv = decode_weight4<C, LEAN>(src, raw[u], iw);
        const float4 (&zv)[C] = raw[u].z;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float z[C], y[C], p[C], gp[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                z[c] = reinterpret_cast<const float*>(&zv[c])[j];
                y[c] = reinterpret_cast<const float*>(&yv[c])[j];
            }
            float w = reinterpret_cast<const float*>(&wv)[j];
            if (src.prob_input) {
#pragma unroll
                for (int c = 0; c < C; ++c) p[c] = z[c];
            } else {
                softmax_c<C>(z, p);
            }
            float dot = 0.0f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                float gc = w * fmaf(a_c[c], y[c], b_c[c]);
                if (w_ce != 0.0f) gc += ce_k * w * y[c] / (p[c] * 0.999f + 5e-4f);
                // d/dp of p*log2(p + eps) = log2(p + eps) + p / ((p + eps) * ln 2)
                if (w_ent != 0.0f) gc += ent_k * (log2f(p[c] + 1e-10f) + p[c] / ((p[c] + 1e-10f) * 0.69314718056f));
                gp[c] = gc;
                dot = fmaf(gc, p[c], dot);
            }
#pragma unroll
            for (int c = 0; c < C; ++c)
                reinterpret_cast<float*>(&ov[c])[j] = src.prob_input ? grad_scale * gp[c] : grad_scale * p[c] * (gp[c] - dot);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) reinterpret_cast<float4*>(dlogits)[(n * C + c) * S4 + s4] = ov[c];
        }
    }
}

// resident blocks per SM of a kernel instantiation (registers decide: 2..4), so that a grid is exactly one wave
template <typename K>
int resident_blocks(K kernel) {
    // all instantiations of one kernel template share a function TYPE, hence this cache: keyed by the function pointer
    static int cached = 0;
    static const void* cached_for = nullptr;
    if (cached == 0 || cached_for != (const void*)kernel) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, kThreads, 0) != cudaSuccess || nb < 1) nb = 1;
        cached = nb > 4 ? 4 : nb;    // every block ends with 6C+3 same-address double atomics: no more than 4 per SM
        cached_for = (const void*)kernel;
    }
    return cached;
}

// blocks per sample: every thread one batch of U groups, capped at `per_sm` resident blocks per SM over the whole grid
int grid_x_for(int64_t s4, int n, int u, int per_sm) {
    int64_t bx = (s4 + (int64_t)kThreads * u - 1) / ((int64_t)kThreads * u);
    int64_t cap = ((int64_t)FPL_NUM_SMS * per_sm + n - 1) / n;
    if (bx > cap) bx = cap;
    return (int)(bx < 1 ? 1 : bx);
}

}  // namespace

#define FPL_DISPATCH_C(C_, ...)                                                     \
    switch (C_) {                                                                   \
        case 2: { constexpr int CC = 2; __VA_ARGS__; } break;                       \
        case 3: { constexpr int CC = 3; __VA_ARGS__; } break;                       \
        case 4: { constexpr int CC = 4; __VA_ARGS__; } break;                       \
        case 5: { constexpr int CC = 5; __VA_ARGS__; } break;                       \
        case 6: { constexpr int CC = 6; __VA_ARGS__; } break;                       \
        case 7: { constexpr int CC = 7; __VA_ARGS__; } break;                       \
        case 8: { constexpr int CC = 8; __VA_ARGS__; } break;                       \
        default: fpl_set_error("class_num %d not in [2,8]", C_); return 2;          \
    }

static int dice_ce_reduce_launch(const float* logits, const LossSrc& src, double* sums, int n, int c, int64_t spatial,
                                 int want_entropy, void* stream) {
    FPL_REQUIRE(spatial % 4 == 0, "fpl_dice_ce_reduce: spatial size %lld must be a multiple of 4", (long long)spatial);
    FPL_REQUIRE(src.soft_y != nullptr || src.label != nullptr, "fpl_dice_ce_reduce: soft_y or label required");
    int64_t s4 = spatial / 4;
    FPL_REQUIRE(n >= 1 && n <= 65535, "fpl_dice_ce_reduce: batch %d not in [1,65535]", n);
    // 4 blocks per SM: every block ends with 6C+3 same-address double atomics, which serialise in L2 (1184 blocks cost
    // ~5 us of a 15 us launch at the configs[2] batch)
    const bool lean = src.soft_y == nullptr && src.weight == nullptr;
    if (c == 2 && lean) {
        // two classes, uint8 inputs: ONE wave of two 256-thread blocks per SM, every thread one batch of up to 8 groups
        // (~140 KB of loads in flight per SM = the bandwidth-delay product: one DRAM round trip per launch)
        fpl_launch(dice_ce_reduce_kernel<2, 8, true>, dim3(grid_x_for(s4, n, 8, resident_blocks(dice_ce_reduce_kernel<2, 8, true>)), n), kThreads, 0,
                   (cudaStream_t)stream, logits, src, sums, n, s4, want_entropy);
    } else if (lean) {
        FPL_DISPATCH_C(c, (fpl_launch(dice_ce_reduce_kernel<CC, (CC <= 5 ? 2 : 1), true>,
                              dim3(grid_x_for(s4, n, CC <= 5 ? 2 : 1, resident_blocks(dice_ce_reduce_kernel<CC, (CC <= 5 ? 2 : 1), true>)), n),
                              kThreads, 0, (cudaStream_t)stream, logits, src, sums, n, s4, want_entropy)));
    } else {
        FPL_DISPATCH_C(c, (fpl_launch(dice_ce_reduce_kernel<CC, 1, false>,
                              dim3(grid_x_for(s4, n, 1, resident_blocks(dice_ce_reduce_kernel<CC, 1, false>)), n),
                              kThreads, 0, (cudaStream_t)stream, logits, src, sums, n, s4, want_entropy)));
    }
    FPL_LAUNCH_CHECK();
    return 0;
}

static int dice_ce_grad_launch(const float* logits, const LossSrc& src, const double* sums, float w_dice, float w_ce,
                               float w_ent, float grad_scale, const float* grad_scale_dev, float* loss, float* dlogits,
                               int n, int c, int64_t spatial, void* stream, int n_global = 0, double* hard_dice = nullptr) {
    FPL_REQUIRE(n_global == 0 || n_global >= n, "fpl_dice_ce_grad: n_global %d < n %d", n_global, n);
    FPL_REQUIRE(spatial % 4 == 0, "fpl_dice_ce_grad: spatial size %lld must be a multiple of 4", (long long)spatial);
    FPL_REQUIRE(src.soft_y != nullptr || src.label != nullptr, "fpl_dice_ce_grad: soft_y or label required");
    int64_t s4 = spatial / 4;
    FPL_REQUIRE(n >= 1 && n <= 65535, "fpl_dice_ce_grad: batch %d not in [1,65535]", n);
    const bool lean = src.soft_y == nullptr && src.weight == nullptr;
    const int gy = dlogits != nullptr ? n : 1;
    if (c == 2 && lean) {
        const dim3 grid(dlogits != nullptr ? grid_x_for(s4, n, 8, resident_blocks(dice_ce_grad_kernel<2, 8, true>)) : 1, gy);
        fpl_launch(dice_ce_grad_kernel<2, 8, true>, grid, kThreads, 0, (cudaStream_t)stream, logits, src, sums, w_dice, w_ce, w_ent,
                   grad_scale, grad_scale_dev, loss, dlogits, n, s4, n_global, hard_dice);
    } else if (lean) {
        FPL_DISPATCH_C(c, (fpl_launch(dice_ce_grad_kernel<CC, (CC <= 5 ? 2 : 1), true>,
                              dim3(dlogits != nullptr ? grid_x_for(s4, n, CC <= 5 ? 2 : 1, 2 * resident_blocks(dice_ce_grad_kernel<CC, (CC <= 5 ? 2 : 1), true>)) : 1, gy),
                              kThreads, 0, (cudaStream_t)stream,
                              logits, src, sums, w_dice, w_ce, w_ent, grad_scale, grad_scale_dev, loss, dlogits, n, s4, n_global, hard_dice)));
    } else {
        FPL_DISPATCH_C(c, (fpl_launch(dice_ce_grad_kernel<CC, 1, false>,
                              dim3(dlogits != nullptr ? grid_x_for(s4, n, 1, 2 * resident_blocks(dice_ce_grad_kernel<CC, 1, false>)) : 1, gy),
                              kThreads, 0, (cudaStream_t)stream,
                              logits, src, sums, w_dice, w_ce, w_ent, grad_scale, grad_scale_dev, loss, dlogits, n, s4, n_global, hard_dice)));
    }
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_dice_ce_reduce(const float* logits, const float* soft_y, const float* weight, double* sums, int n,
                                  int c, int64_t spatial, void* stream) {
    LossSrc src = {soft_y, nullptr, weight, nullptr, nullptr, 0};
    return dice_ce_reduce_launch(logits, src, sums, n, c, spatial, 0, stream);
}

extern "C" int fpl_dice_ce_grad(const float* logits, const float* soft_y, const float* weight, const double* sums,
                                float w_dice, float w_ce, float grad_scale, const float* grad_scale_dev, float* loss,
                                float* dlogits, int n, int c, int64_t spatial, void* stream) {
    LossSrc src = {soft_y, nullptr, weight, nullptr, nullptr, 0};
    return dice_ce_grad_launch(logits, src, sums, w_dice, w_ce, 0.0f, grad_scale, grad_scale_dev, loss, dlogits, n, c,
                               spatial, stream);
}

extern "C" int fpl_dice_ce_reduce_ex(const float* logits, const float* soft_y, const uint8_t* label, const float* weight,
                                     const uint8_t* weight_code, const float* image_weight, double* sums, int n, int c,
                                     int64_t spatial, int want_entropy, int prob_input, void* stream) {
    FPL_REQUIRE(!(prob_input && want_entropy), "fpl_dice_ce_reduce_ex: the entropy term is defined on logits");
    LossSrc src = {soft_y, label, weight, weight_code, image_weight, prob_input};
    return dice_ce_reduce_launch(logits, src, sums, n, c, spatial, want_entropy, stream);
}

extern "C" int fpl_dice_ce_grad_ex(const float* logits, const float* soft_y, const uint8_t* label, const float* weight,
                                   const uint8_t* weight_code, const float* image_weight, const double* sums,
                                   float w_dice, float w_ce, float w_entropy, float grad_scale,
                                   const float* grad_scale_dev, float* loss, float* dlogits, int n, int c,
                                   int64_t spatial, int prob_input, int n_global, void* stream) {
    FPL_REQUIRE(!(prob_input && w_entropy != 0.0f), "fpl_dice_ce_grad_ex: the entropy term is defined on logits");
    LossSrc src = {soft_y, label, weight, weight_code, image_weight, prob_input};
    return dice_ce_grad_launch(logits, src, sums, w_dice, w_ce, w_entropy, grad_scale, grad_scale_dev, loss, dlogits, n,
                               c, spatial, stream, n_global);
}

extern "C" int fpl_dice_ce_loss_ex(const float* logits, const float* soft_y, const uint8_t* label, const float* weight,
                                   const uint8_t* weight_code, const float* image_weight, const double* sums,
                                   float w_dice, float w_ce, float w_entropy, float* loss, double* hard_dice, int n, int c,
                                   int64_t spatial, int prob_input, int n_global, void* stream) {
    FPL_REQUIRE(loss != nullptr, "fpl_dice_ce_loss_ex: loss must not be NULL");
    LossSrc src = {soft_y, label, weight, weight_code, image_weight, prob_input};
    return dice_ce_grad_launch(logits, src, sums, w_dice, w_ce, w_entropy, 1.0f, nullptr, loss, nullptr, n, c, spatial, stream,
                               n_global, hard_dice);
}

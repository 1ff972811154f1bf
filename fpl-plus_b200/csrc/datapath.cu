// Device data path of the training inputs (SURVEY 8 f-3): RandomCrop + RandomFlip of PyMIC's loader
// (PyMIC/pymic/transform/crop.py:170-244, flip.py:14-62) as ONE gather kernel over volumes that stay resident in HBM.
// The host draws the crop origin and the flip axes per sample (same decisions, same order as the reference transforms);
// this kernel cuts the image patch (fp32), the label patch (uint8) and the agreement-code patch (uint8) and applies the
// flips on the fly.  LabelToProbability (one-hot) and NiftyDataset.set_weight_ happen inside the loss kernels
// (fpl_dice_ce_*_ex), so no fp32 one-hot / weight tensor is ever materialised and nothing crosses PCIe per step.
//
// NormalizeWithMeanStd after RandomCrop (PyMIC/pymic/transform/normalize.py, the order of the FPL+ train_transform lists)
// takes its mean / std from each cut patch: patch_stats_kernel writes per-block fp64 partial sums of the source sub-box
// of every sample, and gather_patches_norm_kernel reduces them in a fixed order before it cuts, flips and normalises.
//
// Validation and test volumes (valid_transform / test_transform: NormalizeWithMeanStd and Pad over the whole volume,
// transform/normalize.py, pad.py) go through volume_stats_kernel + pad_normalize_volume_kernel: the same partial-sum walk
// and mean / std prologue, over the source volume or over the padded index space, then one pass that pads (NumPy
// 'reflect', 'edge' when an axis has size 1, labels constant 0) and normalises.
#include <math.h>

#include "common.cuh"
#include "../../include/fplplus_b200.h"

namespace {

struct __align__(16) PatchRow {      // one sample of the batch (64 bytes, built by the host)
    const float* image;              // [C][D][H][W] fp32 (raw or host-normalised, padded to >= patch size)
    const uint8_t* label;            // [D][H][W] or NULL
    const uint8_t* code;             // [D][H][W] agreement code (0/1/2) or NULL
    int D, H, W;
    int d0, h0, w0;                  // crop origin
    int flip;                        // bit 0: depth, bit 1: height, bit 2: width
    int pad[3];
};
static_assert(sizeof(PatchRow) == 64, "PatchRow layout is part of the C ABI (fpl_gather_patches)");

__global__ void __launch_bounds__(256) gather_patches_kernel(const PatchRow* __restrict__ rows, int C, int pd, int ph, int pw,
                                                             float* __restrict__ out_img, uint8_t* __restrict__ out_lab,
                                                             uint8_t* __restrict__ out_code) {
    FPL_PDL_WAIT();
    const int n = blockIdx.y;
    const PatchRow r = rows[n];
    const int64_t pvox = (int64_t)pd * ph * pw;
    const int64_t svox = (int64_t)r.D * r.H * r.W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pvox; i += (int64_t)gridDim.x * blockDim.x) {
        const int w = (int)(i % pw);
        const int64_t t = i / pw;
        const int h = (int)(t % ph), d = (int)(t / ph);
        const int sd = r.d0 + ((r.flip & 1) ? pd - 1 - d : d);
        const int sh = r.h0 + ((r.flip & 2) ? ph - 1 - h : h);
        const int sw = r.w0 + ((r.flip & 4) ? pw - 1 - w : w);
        const int64_t s = ((int64_t)sd * r.H + sh) * r.W + sw;
        for (int c = 0; c < C; ++c) out_img[((int64_t)n * C + c) * pvox + i] = __ldg(r.image + (int64_t)c * svox + s);
        if (out_lab != nullptr) out_lab[(int64_t)n * pvox + i] = r.label != nullptr ? __ldg(r.label + s) : (uint8_t)0;
        if (out_code != nullptr) out_code[(int64_t)n * pvox + i] = r.code != nullptr ? __ldg(r.code + s) : (uint8_t)2;
    }
}

// ---- per-patch NormalizeWithMeanStd ---------------------------------------------------------------------------------
constexpr int kNormMaxC = 16;
constexpr int kNormStats = 5;        // per (sample, block, channel): sum, sum of squares; over the voxels > 0: sum, sum of squares, count
enum NormMode { kNormRaw = 0, kNormFixed = 1, kNormPatch = 2, kNormPatchMasked = 3 };

struct NormParams {
    int mode[kNormMaxC];             // NormMode per channel
    float mean[kNormMaxC];           // kNormFixed only
    float std[kNormMaxC];            // kNormFixed only
};

// blocks per sample of the statistics kernels: a function of the voxel count alone, so the workspace has a closed size and
// the fixed-order reduction of the partials gives the same bits on every run and every SM budget
constexpr int kPatchStatBlocks = 64;     // per patch (a batch has several)
constexpr int kVolumeStatBlocks = 256;   // per whole volume (one launch per volume)
int norm_stat_blocks(int64_t vox, int cap) {
    const int64_t b = (vox + 256 * 8 - 1) / (256 * 8);
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// One block's fp64 partials (sum, sum of squares; over the voxels > 0: sum, sum of squares, count) of one channel over
// the nvox voxels load(i), i in [0, nvox), walked grid-stride; stored to out[0..kNormStats).  No atomics: the caller gives
// every block its own slots.  nvox <= 2^30, so i + grid stride stays in int.
template <class Load>
__device__ __forceinline__ void block_norm_partials(int nvox, int mode, Load load, double (*s_red)[kNormStats],
                                                    double* __restrict__ out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double acc[kNormStats] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvox; i += gridDim.x * blockDim.x) {
        const double v = (double)load(i);
        acc[0] += v;
        acc[1] = fma(v, v, acc[1]);
        if (mode == kNormPatchMasked && v > 0.0) {
            acc[2] += v;
            acc[3] = fma(v, v, acc[3]);
            acc[4] += 1.0;
        }
    }
#pragma unroll
    for (int k = 0; k < kNormStats; ++k) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kNormStats; ++k) s_red[warp][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < kNormStats) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_red[w][threadIdx.x];
        out[threadIdx.x] = t;
    }
    __syncthreads();
}

// Per-channel mean / std into shared memory (warp per channel, partials part[nb][C][kNormStats] reduced in a fixed order),
// with the rules of datapath.normalize_with_mean_std: population std floored at 1e-8; masked statistics from the voxels
// > 0, from all nvox voxels when there are none.  Raw channels get (0, 1) and are not read.  The caller syncs the block.
__device__ __forceinline__ void norm_mean_std(const NormParams& P, int C, const double* __restrict__ part, int nb,
                                              double nvox, float* s_mean, float* s_std) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int c = warp; c < C; c += 8) {
        float mean = 0.f, stdv = 1.f;
        if (P.mode[c] == kNormFixed) {
            mean = P.mean[c];
            stdv = P.std[c];
        } else if (P.mode[c] >= kNormPatch) {
            double acc[kNormStats] = {0.0, 0.0, 0.0, 0.0, 0.0};
            for (int b = lane; b < nb; b += 32) {
                const double* p = part + ((int64_t)b * C + c) * kNormStats;
#pragma unroll
                for (int k = 0; k < kNormStats; ++k) acc[k] += p[k];
            }
#pragma unroll
            for (int k = 0; k < kNormStats; ++k) {
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
            }
            double cnt = nvox, sum = acc[0], sq = acc[1];
            if (P.mode[c] == kNormPatchMasked && acc[4] > 0.0) {
                cnt = acc[4];
                sum = acc[2];
                sq = acc[3];
            }
            const double m = sum / cnt;
            mean = (float)m;
            stdv = (float)fmax(sqrt(fmax(sq / cnt - m * m, 0.0)), 1e-8);
        }
        if (lane == 0) {
            s_mean[c] = mean;
            s_std[c] = stdv;
        }
    }
}

// Grid (blocks, n).  Flips do not change sums, so the block walks the unflipped source sub-box of its sample.  No atomics:
// every block stores its own partials (part[n][block][C][kNormStats]; the slots of other channels are left unwritten).
__global__ void __launch_bounds__(256) patch_stats_kernel(const PatchRow* __restrict__ rows, int C, int pd, int ph, int pw,
                                                          NormParams P, double* __restrict__ part) {
    FPL_PDL_WAIT();
    __shared__ double s_red[8][kNormStats];
    const int n = blockIdx.y;
    const PatchRow r = rows[n];
    const int64_t svox = (int64_t)r.D * r.H * r.W;
    for (int c = 0; c < C; ++c) {
        const int mode = P.mode[c];
        if (mode < kNormPatch) continue;
        const float* src = r.image + (int64_t)c * svox;
        block_norm_partials(
            pd * ph * pw, mode,
            [&](int i) {
                const int w = i % pw, t = i / pw;
                const int h = t % ph, d = t / ph;
                return __ldg(src + ((int64_t)(r.d0 + d) * r.H + r.h0 + h) * r.W + r.w0 + w);
            },
            s_red, part + (((int64_t)n * gridDim.x + blockIdx.x) * C + c) * kNormStats);
    }
    FPL_PDL_TRIGGER();               // after this block's partials are stored
}

// gather_patches_kernel with (x - mean) / std applied to the normalised channels.  The prologue (norm_mean_std) turns the
// partials of the sample into mean / std.
__global__ void __launch_bounds__(256) gather_patches_norm_kernel(const PatchRow* __restrict__ rows, int C, int pd, int ph,
                                                                  int pw, NormParams P, const double* __restrict__ part,
                                                                  int nb, float* __restrict__ out_img,
                                                                  uint8_t* __restrict__ out_lab,
                                                                  uint8_t* __restrict__ out_code) {
    FPL_PDL_WAIT();
    __shared__ float s_mean[kNormMaxC], s_std[kNormMaxC];
    const int n = blockIdx.y;
    const int pvox = pd * ph * pw;   // <= 2^30 (checked by the launcher): i + grid stride stays in int
    norm_mean_std(P, C, part + (int64_t)n * nb * C * kNormStats, nb, (double)pvox, s_mean, s_std);
    __syncthreads();
    const PatchRow r = rows[n];
    const int64_t svox = (int64_t)r.D * r.H * r.W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < pvox; i += gridDim.x * blockDim.x) {
        const int w = i % pw, t = i / pw;
        const int h = t % ph, d = t / ph;
        const int sd = r.d0 + ((r.flip & 1) ? pd - 1 - d : d);
        const int sh = r.h0 + ((r.flip & 2) ? ph - 1 - h : h);
        const int sw = r.w0 + ((r.flip & 4) ? pw - 1 - w : w);
        const int64_t s = ((int64_t)sd * r.H + sh) * r.W + sw;
        for (int c = 0; c < C; ++c) {
            float v = __ldg(r.image + (int64_t)c * svox + s);
            if (P.mode[c] != kNormRaw) v = (v - s_mean[c]) / s_std[c];
            out_img[((int64_t)n * C + c) * pvox + i] = v;
        }
        if (out_lab != nullptr) out_lab[(int64_t)n * pvox + i] = r.label != nullptr ? __ldg(r.label + s) : (uint8_t)0;
        if (out_code != nullptr) out_code[(int64_t)n * pvox + i] = r.code != nullptr ? __ldg(r.code + s) : (uint8_t)2;
    }
}

// ---- whole-volume Pad + NormalizeWithMeanStd (validation / test inputs) ----------------------------------------------
struct PadGeom {
    int D, H, W;                     // source volume
    int oD, oH, oW;                  // padded volume (>= the source per axis)
    int lo_d, lo_h, lo_w;            // lower margins (o - n) / 2, as datapath.pad_to
    int edge;                        // 1: NumPy 'edge' (pad_to's choice when an axis has size 1), 0: 'reflect'
};

// Source index of padded index p along an axis of n voxels: NumPy 'reflect' (mirror without repeating the edge voxel; for
// margins > n - 1 NumPy reflects again, so the index is periodic with period 2(n - 1)), or 'edge' (clamp).  Reflect needs
// n >= 2, which the edge rule guarantees.
__device__ __forceinline__ int pad_source_index(int p, int n, int edge) {
    if (p >= 0 && p < n) return p;
    if (edge) return p < 0 ? 0 : n - 1;
    const int period = 2 * (n - 1);
    int m = p % period;
    if (m < 0) m += period;
    return m < n ? m : period - m;
}

__device__ __forceinline__ int64_t pad_source_offset(const PadGeom& g, int i, bool* inside) {
    const int w = i % g.oW, t = i / g.oW;
    const int h = t % g.oH, d = t / g.oH;
    const int pd = d - g.lo_d, ph = h - g.lo_h, pw = w - g.lo_w;
    *inside = (unsigned)pd < (unsigned)g.D && (unsigned)ph < (unsigned)g.H && (unsigned)pw < (unsigned)g.W;
    return ((int64_t)pad_source_index(pd, g.D, g.edge) * g.H + pad_source_index(ph, g.H, g.edge)) * g.W +
           pad_source_index(pw, g.W, g.edge);
}

// Grid (blocks).  Partials part[block][C][kNormStats] of the statistics channels over the source volume, or (padded) over
// the padded index space walked through the pad map, without materialising the padded volume.
__global__ void __launch_bounds__(256) volume_stats_kernel(const float* __restrict__ img, int C, PadGeom g, int padded,
                                                           NormParams P, double* __restrict__ part) {
    FPL_PDL_WAIT();
    __shared__ double s_red[8][kNormStats];
    const int64_t svox = (int64_t)g.D * g.H * g.W;
    for (int c = 0; c < C; ++c) {
        const int mode = P.mode[c];
        if (mode < kNormPatch) continue;
        const float* src = img + (int64_t)c * svox;
        double* out = part + ((int64_t)blockIdx.x * C + c) * kNormStats;
        if (padded) {
            block_norm_partials(
                g.oD * g.oH * g.oW, mode,
                [&](int i) {
                    bool inside;
                    return __ldg(src + pad_source_offset(g, i, &inside));
                },
                s_red, out);
        } else {
            block_norm_partials((int)svox, mode, [&](int i) { return __ldg(src + i); }, s_red, out);
        }
    }
    FPL_PDL_TRIGGER();               // after this block's partials are stored
}

// Grid-stride over the padded volume: image through the pad map and (x - mean) / std of the normalised channels; label
// with constant 0 outside the source box.
__global__ void __launch_bounds__(256) pad_normalize_volume_kernel(const float* __restrict__ img,
                                                                   const uint8_t* __restrict__ lab, int C, PadGeom g,
                                                                   NormParams P, const double* __restrict__ part, int nb,
                                                                   double stat_vox, float* __restrict__ out_img,
                                                                   uint8_t* __restrict__ out_lab) {
    FPL_PDL_WAIT();
    __shared__ float s_mean[kNormMaxC], s_std[kNormMaxC];
    norm_mean_std(P, C, part, nb, stat_vox, s_mean, s_std);
    __syncthreads();
    const int ovox = g.oD * g.oH * g.oW;   // <= 2^30 (checked by the launcher): i + grid stride stays in int
    const int64_t svox = (int64_t)g.D * g.H * g.W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ovox; i += gridDim.x * blockDim.x) {
        bool inside;
        const int64_t s = pad_source_offset(g, i, &inside);
        for (int c = 0; c < C; ++c) {
            float v = __ldg(img + (int64_t)c * svox + s);
            if (P.mode[c] != kNormRaw) v = (v - s_mean[c]) / s_std[c];
            out_img[(int64_t)c * ovox + i] = v;
        }
        if (out_lab != nullptr) out_lab[i] = inside ? __ldg(lab + s) : (uint8_t)0;
    }
}

// Host side of both normalising entry points: per-channel modes / fixed values -> NormParams, with the same checks.
int norm_params_from_host(const char* fn, int c, const int* h_mode, const float* h_mean, const float* h_std, NormParams* P,
                          bool* stats) {
    *P = NormParams{};
    *stats = false;
    for (int i = 0; i < c; ++i) {
        FPL_REQUIRE(h_mode[i] >= kNormRaw && h_mode[i] <= kNormPatchMasked, "%s: channel %d: mode %d", fn, i, h_mode[i]);
        P->mode[i] = h_mode[i];
        if (h_mode[i] == kNormFixed) {
            FPL_REQUIRE(h_mean != nullptr && h_std != nullptr, "%s: channel %d: fixed mode needs mean and std", fn, i);
            FPL_REQUIRE(h_std[i] > 0.f && isfinite(h_std[i]) && isfinite(h_mean[i]), "%s: channel %d: mean %g / std %g", fn,
                        i, h_mean[i], h_std[i]);
            P->mean[i] = h_mean[i];
            P->std[i] = h_std[i];
        }
        *stats = *stats || h_mode[i] >= kNormPatch;
    }
    return 0;
}

}  // namespace

extern "C" int fpl_gather_patches(const void* d_rows, int n, int c, int pd, int ph, int pw, float* out_image,
                                  uint8_t* out_label, uint8_t* out_code, void* stream) {
    FPL_REQUIRE(n >= 1 && n <= 65535 && c >= 1 && pd >= 1 && ph >= 1 && pw >= 1, "fpl_gather_patches: bad sizes");
    FPL_REQUIRE(d_rows != nullptr && out_image != nullptr, "fpl_gather_patches: NULL argument");
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(d_rows) & 15) == 0, "fpl_gather_patches: table must be 16-byte aligned");
    const int64_t pvox = (int64_t)pd * ph * pw;
    int bx = (int)((pvox + 256 * 4 - 1) / (256 * 4));
    if (bx > FPL_NUM_SMS * 4) bx = FPL_NUM_SMS * 4;
    if (bx < 1) bx = 1;
    fpl_launch(gather_patches_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, reinterpret_cast<const PatchRow*>(d_rows), c, pd,
               ph, pw, out_image, out_label, out_code);
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t fpl_gather_patches_norm_workspace_bytes(int n, int c, int pd, int ph, int pw) {
    if (n < 1 || c < 1 || pd < 1 || ph < 1 || pw < 1) return -1;
    return (int64_t)n * norm_stat_blocks((int64_t)pd * ph * pw, kPatchStatBlocks) * c * kNormStats * (int64_t)sizeof(double);
}

extern "C" int fpl_gather_patches_norm(const void* d_rows, int n, int c, int pd, int ph, int pw, const int* h_mode,
                                       const float* h_mean, const float* h_std, void* workspace, int64_t workspace_bytes,
                                       float* out_image, uint8_t* out_label, uint8_t* out_code, void* stream) {
    FPL_REQUIRE(n >= 1 && n <= 65535 && c >= 1 && pd >= 1 && ph >= 1 && pw >= 1, "fpl_gather_patches_norm: bad sizes");
    FPL_REQUIRE((int64_t)pd * ph * pw <= (1 << 30), "fpl_gather_patches_norm: patch of more than 2^30 voxels");
    FPL_REQUIRE(c <= kNormMaxC, "fpl_gather_patches_norm: %d channels, at most %d", c, kNormMaxC);
    FPL_REQUIRE(d_rows != nullptr && out_image != nullptr && h_mode != nullptr, "fpl_gather_patches_norm: NULL argument");
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(d_rows) & 15) == 0, "fpl_gather_patches_norm: table must be 16-byte aligned");
    NormParams P;
    bool stats;
    const int rc = norm_params_from_host("fpl_gather_patches_norm", c, h_mode, h_mean, h_std, &P, &stats);
    if (rc != 0) return rc;
    const int64_t pvox = (int64_t)pd * ph * pw;
    const int nb = norm_stat_blocks(pvox, kPatchStatBlocks);
    if (stats) {
        FPL_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0,
                    "fpl_gather_patches_norm: workspace must be 8-byte aligned");
        FPL_REQUIRE(workspace_bytes >= fpl_gather_patches_norm_workspace_bytes(n, c, pd, ph, pw),
                    "fpl_gather_patches_norm: workspace of %lld bytes, needs %lld", (long long)workspace_bytes,
                    (long long)fpl_gather_patches_norm_workspace_bytes(n, c, pd, ph, pw));
        fpl_launch(patch_stats_kernel, dim3(nb, n), 256, 0, (cudaStream_t)stream, reinterpret_cast<const PatchRow*>(d_rows),
                   c, pd, ph, pw, P, reinterpret_cast<double*>(workspace));
        FPL_LAUNCH_CHECK();
    }
    int bx = (int)((pvox + 256 * 4 - 1) / (256 * 4));
    if (bx > FPL_NUM_SMS * 4) bx = FPL_NUM_SMS * 4;
    if (bx < 1) bx = 1;
    fpl_launch(gather_patches_norm_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, reinterpret_cast<const PatchRow*>(d_rows),
               c, pd, ph, pw, P, reinterpret_cast<const double*>(workspace), nb, out_image, out_label, out_code);
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t fpl_pad_normalize_volume_workspace_bytes(int c, int d, int h, int w, int od, int oh, int ow) {
    if (c < 1 || d < 1 || h < 1 || w < 1 || od < d || oh < h || ow < w) return -1;
    return (int64_t)norm_stat_blocks((int64_t)od * oh * ow, kVolumeStatBlocks) * c * kNormStats * (int64_t)sizeof(double);
}

extern "C" int fpl_pad_normalize_volume(const float* image, const uint8_t* label, int c, int d, int h, int w, int od, int oh,
                                        int ow, const int* h_mode, const float* h_mean, const float* h_std,
                                        int stats_after_pad, void* workspace, int64_t workspace_bytes, float* out_image,
                                        uint8_t* out_label, void* stream) {
    FPL_REQUIRE(c >= 1 && d >= 1 && h >= 1 && w >= 1 && od >= d && oh >= h && ow >= w,
                "fpl_pad_normalize_volume: bad sizes (%d x %d x %d x %d padded to %d x %d x %d)", c, d, h, w, od, oh, ow);
    FPL_REQUIRE((int64_t)od * oh * ow <= (1 << 30), "fpl_pad_normalize_volume: volume of more than 2^30 voxels");
    FPL_REQUIRE(c <= kNormMaxC, "fpl_pad_normalize_volume: %d channels, at most %d", c, kNormMaxC);
    FPL_REQUIRE(image != nullptr && out_image != nullptr && h_mode != nullptr, "fpl_pad_normalize_volume: NULL argument");
    FPL_REQUIRE((label == nullptr) == (out_label == nullptr), "fpl_pad_normalize_volume: give both label and out_label, or neither");
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(image) & 3) == 0 && (reinterpret_cast<uintptr_t>(out_image) & 3) == 0,
                "fpl_pad_normalize_volume: image buffers must be 4-byte aligned");
    FPL_REQUIRE(stats_after_pad == 0 || stats_after_pad == 1, "fpl_pad_normalize_volume: stats_after_pad %d", stats_after_pad);
    NormParams P;
    bool stats;
    const int rc = norm_params_from_host("fpl_pad_normalize_volume", c, h_mode, h_mean, h_std, &P, &stats);
    if (rc != 0) return rc;
    PadGeom g;
    g.D = d, g.H = h, g.W = w, g.oD = od, g.oH = oh, g.oW = ow;
    g.lo_d = (od - d) / 2, g.lo_h = (oh - h) / 2, g.lo_w = (ow - w) / 2;
    g.edge = (d == 1 || h == 1 || w == 1) ? 1 : 0;
    const int64_t ovox = (int64_t)od * oh * ow;
    const int64_t stat_vox = stats_after_pad ? ovox : (int64_t)d * h * w;
    const int nb = norm_stat_blocks(stat_vox, kVolumeStatBlocks);
    if (stats) {
        FPL_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0,
                    "fpl_pad_normalize_volume: workspace must be 8-byte aligned");
        const int64_t need = fpl_pad_normalize_volume_workspace_bytes(c, d, h, w, od, oh, ow);
        FPL_REQUIRE(workspace_bytes >= need, "fpl_pad_normalize_volume: workspace of %lld bytes, needs %lld",
                    (long long)workspace_bytes, (long long)need);
        fpl_launch(volume_stats_kernel, dim3(nb), 256, 0, (cudaStream_t)stream, image, c, g, stats_after_pad, P,
                   reinterpret_cast<double*>(workspace));
        FPL_LAUNCH_CHECK();
    }
    int bx = (int)((ovox + 256 * 4 - 1) / (256 * 4));
    if (bx > FPL_NUM_SMS * 4) bx = FPL_NUM_SMS * 4;
    if (bx < 1) bx = 1;
    fpl_launch(pad_normalize_volume_kernel, dim3(bx), 256, 0, (cudaStream_t)stream, image, label, c, g, P,
               reinterpret_cast<const double*>(stats ? workspace : nullptr), nb, (double)stat_vox, out_image, out_label);
    FPL_LAUNCH_CHECK();
    return 0;
}

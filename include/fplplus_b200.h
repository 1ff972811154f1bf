/*
 * fplplus_b200 -- C ABI of the B200-native FPL+ hot path (sm_100a).
 *
 * The reference (HiLab-git/FPL-plus) is pure Python and has no FFI; every entry
 * point below replaces the torch/NumPy call sequence named in its comment
 * (paths relative to the reference tree).  INTEGRATION.md shows the ctypes
 * binding a PyMIC maintainer would add.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless named h_*; the caller owns them.
 *   - `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, non-zero on error; fpl_last_error()
 *     returns a thread-local message.  Nothing here falls back to the CPU.
 *   - activations use the "C8-planar" layout  [N][D][C/8][H][W][8]  in bf16
 *     (channel groups of 8 are 16-byte vectors; a tensor that is a channel slice
 *     of a wider buffer -- e.g. one half of a skip/up concat buffer -- is
 *     addressed by (base, c8_total, c8_offset)).  Images/logits at the PyMIC
 *     boundary stay NCDHW fp32.
 */
#ifndef FPLPLUS_B200_H
#define FPLPLUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* fpl_last_error(void);
int fpl_version(void);
/* Number of SMs the persistent kernels size their grids for (default 148).  One process per GPU with overlapped NCCL
 * all-reduces (agent_seg.py:695 is nn.DataParallel in the reference) sets 148 - NCCL_MAX_CTAS so that the communication
 * kernels and the statically tiled conv kernels never queue behind each other. */
int fpl_set_sm_budget(int sms);
/* Number of kernels this library has launched in the process so far (reset != 0 zeroes it).
 * Instrumentation only (bench.py reports it as "gpu_launches"); no reference counterpart. */
long long fpl_launch_count(int reset);
/* 1 when the running device is sm_100 (tcgen05 kernels usable), else 0. */
int fpl_device_is_sm100(void);

/* ---- (a) conv3d: PyMIC/pymic/net/net3d/unet2d5_dsbn.py:75,79 (nn.Conv3d k3 p1 / k(1,3,3) p(0,1,1)) ---- */

/* Bytes of the staged bf16 weight image fpl_conv3d_prep_weight writes. */
int64_t fpl_conv3d_weight_image_bytes(int cin, int cout, int kd);
/* fp32 [Cout][Cin][kd][3][3] -> staged bf16 image for the tcgen05 kernel.
 * transpose_flip=0: forward operand.  =1: dgrad operand (taps flipped, Cin/Cout
 * swapped; `cin`/`cout` are still those of the FORWARD conv). */
int fpl_conv3d_prep_weight(const float* w, int cin, int cout, int kd, int transpose_flip,
                           void* image, void* stream);
/* The same for `count` (<= 80) convolutions in ONE launch; all arrays are HOST arrays of length count
 * (w / images hold device pointers). */
int fpl_conv3d_prep_weight_batch(int count, const float* const* h_w, const int* h_cin, const int* h_cout,
                                 const int* h_kd, const int* h_transpose_flip, void* const* h_images, void* stream);
/* Implicit-GEMM conv on tcgen05/TMEM fed by TMA.  x: C8-planar bf16 with
 * `cin` channels at (x_c8tot, x_c8off); y likewise with `cout` channels.
 * bias may be NULL.  stats (double[2*cout]: sum, sum of squares of the fp32
 * results incl. bias) may be NULL; it is ACCUMULATED into (caller zeroes).
 * `image` must have been prepared for (cin, cout) of THIS call (for dgrad call
 * with cin=Cout_fwd, cout=Cin_fwd and the transpose_flip image). */
int fpl_conv3d_tc(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias,
                  void* y, int y_c8tot, int y_c8off, double* stats,
                  int n, int d, int h, int w, int cin, int cout, int kd, void* stream);
/* Depth-folded variant for the small-channel k3 layers (csrc/conv_tc_dfold.cu): every input plane tile issues 9 MMAs
 * of N = 3*Cout into the accumulators of the three output planes it feeds, with all 27 weight taps resident in
 * shared memory.  Same contract as fpl_conv3d_tc (kd = 3 only); its own staged image.  image_bytes returns -1 when
 * (cin, cout) is not eligible (needs cin <= 64, cout in {16,32,64}, 27*cin*cout*2 B <= 112 KB). */
int64_t fpl_conv3d_dfold_image_bytes(int cin, int cout);
int fpl_conv3d_dfold_prep_weight(const float* w, int cin, int cout, int transpose_flip, void* image, void* stream);
int fpl_conv3d_dfold_prep_weight_batch(int count, const float* const* h_w, const int* h_cin, const int* h_cout,
                                       const int* h_transpose_flip, void* const* h_images, void* stream);
int fpl_conv3d_tc_dfold(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias,
                        void* y, int y_c8tot, int y_c8off, double* stats,
                        int n, int d, int h, int w, int cin, int cout, void* stream);
/* k = (3,1,1) conv (depth taps only) and its wgrad on the same kernels with ONE in-plane tap; w / dW are fp32
 * [Cout][Cin][3].  With fpl_patch9_c8 (1-channel fp32 image -> 16 bf16 channels holding the 9 in-plane neighbours)
 * they run the stem conv k(3,3,3), in_chns = 1 (unet2d5_dsbn.py:75, first conv3d_1) on the tensor cores. */
/* split_hi_lo != 0: 32 channels, the second 16 hold the bf16 rounding residual x - bf16(x) (hi + lo = 16 mantissa
 * bits); fpl_conv3d_tc_k311 with cin = 48 weights [w_hi | w_hi | w_lo] and a_channels = 32 (the third K block reads
 * the hi channels again) then evaluates x*w to ~2^-16 although every operand is bf16. */
int fpl_patch9_c8(const float* x, void* out, int split_hi_lo, int n, int d, int h, int w, void* stream);
int fpl_conv3d_k311_prep_weight(const float* w, int cin, int cout, void* image, void* stream);
int fpl_conv3d_tc_k311(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias,
                       void* y, int y_c8tot, int y_c8off, double* stats,
                       int n, int d, int h, int w, int cin, int cout, int a_channels, void* stream);
int fpl_conv3d_wgrad_tc_k311(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                             float* dw, int n, int d, int h, int w, int cin, int cout, void* stream);
/* CUDA-core conv with the same contract (used for shapes the tensor kernel does
 * not cover and as the on-device cross-check).  w is fp32 [Cout][Cin][kd][3][3];
 * transpose_flip as above; round_w_bf16!=0 rounds weights to bf16 first. */
int fpl_conv3d_direct(const void* x, int x_c8tot, int x_c8off, const float* w, const float* bias,
                      void* y, int y_c8tot, int y_c8off, double* stats,
                      int n, int d, int h, int w_, int cin, int cout, int kd,
                      int transpose_flip, int round_w_bf16, void* stream);
/* wgrad: dW[Cout][Cin][kd][3][3] (fp32, ACCUMULATED into) = sum_v dy[v] (x) x[v+tap]. */
int fpl_conv3d_wgrad(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                     float* dw, int n, int d, int h, int w, int cin, int cout, int kd, void* stream);

/* The same contract on tcgen05 (both operands MN-major straight from the C8-planar layout, the 9
 * in-plane taps as shifted descriptors of one TMA-staged halo tile, accumulators resident in TMEM over
 * the CTA's whole split-K slice).  Needs cin % 8 == 0 and cout % 16 == 0. */
int fpl_conv3d_wgrad_tc(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                        float* dw, int n, int d, int h, int w, int cin, int cout, int kd, void* stream);

/* Tap-major variant: scratch S[kd*9+t9][cout][cin] (fp32, ACCUMULATED into) so that the epilogue's atomics are
 * coalesced; fpl_wgrad_tapmajor_to_dw_batch then folds the scratch of up to 64 layers into the PyTorch layout
 * (dW[co][ci][tap] += S[tap][co][ci], co < cout) in one launch; all arrays are HOST arrays of length count;
 * h_scratch_cout (may be NULL = h_cout) is the number of output-channel rows the scratch was computed with (the head:
 * classes padded to 8, only the real classes are folded). */
int fpl_conv3d_wgrad_tc_tapmajor(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                                 float* scratch, int n, int d, int h, int w, int cin, int cout, int kd, void* stream);
int fpl_wgrad_tapmajor_to_dw_batch(int count, const float* const* h_scratch, float* const* h_dw, const int* h_cout,
                                   const int* h_cin, const int* h_taps, const int* h_scratch_cout, void* stream);

/* Adds segments of one backward pass's flat gradient buffer into the network's master gradient buffer (the storage
 * behind every p.grad) in one launch: replaces autograd's per-parameter AccumulateGrad adds when the source and the
 * target batch of a training_all step (agent_seg.py:459-495) go through the same weights.  d_table is a DEVICE array
 * [segments][3] = {src offset, dst offset, count} in floats, offsets multiples of 4; the adds are atomic (the two
 * passes run on two streams).  max_numel = the largest count (grid sizing). */
int fpl_grad_scatter_add(float* dst, const float* src, const int* d_table, int segments, int max_numel, void* stream);

/* ---- device data path of the training inputs: RandomCrop + RandomFlip (transform/crop.py:170-244, flip.py:14-62) -----
 * d_rows: DEVICE table of n rows of 64 bytes
 *   { const float* image [C][D][H][W]; const uint8_t* label [D][H][W] or NULL; const uint8_t* code [D][H][W] or NULL;
 *     int32 D, H, W; int32 d0, h0, w0 (crop origin); int32 flip (bit 0 depth, 1 height, 2 width); int32 pad[3] }
 * of volumes resident in HBM.  Writes the batch: out_image fp32 [n][C][pd][ph][pw], out_label uint8 [n][pd][ph][pw]
 * (may be NULL), out_code uint8 [n][pd][ph][pw] (may be NULL; a sample without a code map gets 2 = weight 1).
 * out[d,h,w] = volume[d0 + (flip_d ? pd-1-d : d), h0 + (flip_h ? ph-1-h : h), w0 + (flip_w ? pw-1-w : w)].
 * LabelToProbability and set_weight_ follow inside fpl_dice_ce_*_ex. */
int fpl_gather_patches(const void* d_rows, int n, int c, int pd, int ph, int pw, float* out_image,
                       uint8_t* out_label, uint8_t* out_code, void* stream);

/* fpl_gather_patches followed by NormalizeWithMeanStd of each cut patch (transform/normalize.py applied after RandomCrop).
 * h_mode, h_mean, h_std: HOST arrays of c entries (c <= 16).  h_mode[i]: 0 = channel i is copied raw; 1 = (x - h_mean[i]) /
 * h_std[i]; 2 = mean / population std of the channel over the patch; 3 = the same over the patch's voxels > 0 (over the
 * whole patch when it has none).  The std of modes 2 / 3 is floored at 1e-8; h_mean / h_std are read for mode 1 only
 * (may be NULL otherwise).  The statistics are fp64 sums written per block into `workspace` (8-byte aligned, at least
 * fpl_gather_patches_norm_workspace_bytes(n, c, pd, ph, pw) bytes; may be NULL when no channel has mode 2 or 3) and
 * reduced in a fixed order, so the batch is bitwise reproducible.  Label and code outputs as fpl_gather_patches. */
int64_t fpl_gather_patches_norm_workspace_bytes(int n, int c, int pd, int ph, int pw);
int fpl_gather_patches_norm(const void* d_rows, int n, int c, int pd, int ph, int pw, const int* h_mode, const float* h_mean,
                            const float* h_std, void* workspace, int64_t workspace_bytes, float* out_image,
                            uint8_t* out_label, uint8_t* out_code, void* stream);

/* ---- optimiser: torch.optim.Adam(params, lr, weight_decay=wd) of net_run/get_optimizer.py:16-17 (coupled L2) ----------
 * ONE launch over all tensors.  d_segs: DEVICE table of nseg rows of 48 bytes
 *   { float* param; const float* grad; float* exp_avg; float* exp_avg_sq; float* step; int32 numel; int32 pad }
 * (all pointers 16-byte aligned); d_chunks: DEVICE int32 [nchunks][2] = {row, first element}, one entry per
 * fpl_adam_chunk_elems() elements of every tensor.  step is torch's per-parameter step counter (fp32, incremented here
 * after the update); the learning rate is *lr_dev when lr_dev != NULL (CUDA-graph replays under MultiStepLR,
 * get_optimizer.py:50-54), else lr_host.  Hyper-parameters are doubles: torch evaluates 1 - beta, beta^step and
 * lr / bias_correction in double and rounds the results to fp32.  d_done_counter: DEVICE uint32 zero-initialised once by the caller. */
int fpl_adam_multi_tensor(const void* d_segs, int nseg, const int* d_chunks, int nchunks, const float* lr_dev,
                          double lr_host, double beta1, double beta2, double eps, double weight_decay,
                          unsigned int* d_done_counter, void* stream);
int fpl_adam_chunk_elems(void);

/* ---- inference epilogue: eval-mode BatchNorm + PReLU + Dropout folded into the conv kernels --------------------------
 * In eval mode nn.BatchNorm3d is the per-channel affine map of the running statistics (dsbn.py:54-57), so
 * conv -> BN -> PReLU -> Dropout (unet2d5_dsbn.py:75-81) is  a = dropout(prelu(acc * scale + shift))  with
 * scale = gamma / sqrt(running_var + eps), shift = beta + (conv bias - running_mean) * scale: the conv epilogue writes the
 * activation and the fpl_dsbn_act_fwd pass (4 B/element of HBM traffic per layer) disappears from no-grad forwards.
 * fpl_dsbn_eval_affine_batch computes scale / shift of up to 48 layers in one launch (HOST arrays of DEVICE pointers). */
int fpl_dsbn_eval_affine_batch(int count, const float* const* h_gamma, const float* const* h_beta,
                               const float* const* h_running_mean, const float* const* h_running_var,
                               const float* const* h_conv_bias, float* const* h_scale, float* const* h_shift,
                               const int* h_c, float eps, void* stream);
int fpl_conv3d_tc_act(const void* x, int x_c8tot, int x_c8off, const void* image, void* a, int a_c8tot, int a_c8off,
                      int n, int d, int h, int w, int cin, int cout, int kd, const float* scale, const float* shift,
                      const float* slope, float drop_p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                      void* stream);
int fpl_conv3d_tc_dfold_act(const void* x, int x_c8tot, int x_c8off, const void* image, void* a, int a_c8tot, int a_c8off,
                            int n, int d, int h, int w, int cin, int cout, const float* scale, const float* shift,
                            const float* slope, void* stream);
int fpl_conv3d_tc_k311_act(const void* x, int x_c8tot, int x_c8off, const void* image, void* a, int a_c8tot, int a_c8off,
                           int n, int d, int h, int w, int cin, int cout, int a_channels, const float* scale,
                           const float* shift, const float* slope, void* stream);

/* nn.MaxPool3d((pool_kd,2,2)) (unet2d5_dsbn.py:104-117) of a C8-planar activation that the inference epilogue already
 * wrote; no argmax codes (no-grad forwards only). */
int fpl_maxpool_c8(const void* a, int a_c8tot, int a_c8off, void* pooled, int p_c8tot, int p_c8off, int pool_kd,
                   int n, int d, int h, int w, int c, void* stream);

/* The (1,3,3) output conv (unet2d5_dsbn.py:301-308) on CUDA cores, one thread per voxel (csrc/head.cu); cin = 16 or 32,
 * class_num <= 8, w fp32 [classes][cin][1][3][3].
 * fpl_head_fwd  : logits fp32 NCDHW = conv(x) + bias.
 * fpl_head_dgrad: g = gradient wrt x (C8-planar bf16) from dlogits fp32 NCDHW; the same pass writes dl8 (may be NULL), the
 *                 bf16 copy of dlogits with the classes padded to one channel group that the tensor-core wgrad reads, and
 *                 ACCUMULATES the bias gradient dbias[classes] (may be NULL). */
int fpl_head_fwd(const void* x, int x_c8tot, int x_c8off, const float* w, const float* bias, float* logits, int n, int d,
                 int h, int w_, int cin, int classes, void* stream);
int fpl_head_dgrad(const float* dlogits, const float* w, void* g, int g_c8tot, int g_c8off, void* dl8, int dl_c8tot,
                   int dl_c8off, float* dbias, int n, int d, int h, int w_, int cin, int classes, void* stream);

/* UpBlock in `bilinear = True` mode (unet2d5_dsbn.py:149-150, 170-176): 1x1 conv (run as a (1,3,3) conv whose off-centre
 * taps are zero, on the ordinary conv kernels) followed by nn.Upsample(scale_factor=2, trilinear / bilinear,
 * align_corners=True).  (n, d, h, w) is the LOW-resolution geometry; kd2 = 2 interpolates depth too (3-D blocks),
 * kd2 = 1 in-plane only (2-D blocks).  The backward form gathers (deterministic). */
int fpl_upsample2x_c8(const void* x, int x_c8tot, int x_c8off, void* y, int y_c8tot, int y_c8off, int n, int d, int h, int w,
                      int c, int kd2, void* stream);
int fpl_upsample2x_c8_bwd(const void* gy, int gy_c8tot, int gy_c8off, void* gx, int gx_c8tot, int gx_c8off, int n, int d,
                          int h, int w, int c, int kd2, void* stream);
/* out[c] += sum over voxels of g[., c] (bias gradient from a C8-planar output gradient). */
int fpl_channel_sum_c8(const void* g, int g_c8tot, int g_c8off, float* out, int n, int d, int h, int w, int c, void* stream);

/* stem: image fp32 NCDHW (in_chns <= 8) -> C8-planar bf16, conv k3 p1 + bias + stats. */
int fpl_stem_conv_fwd(const float* x, const float* w, const float* bias, void* y, int y_c8tot, int y_c8off,
                      double* stats, int n, int cin, int d, int h, int w_, int cout, int kd, void* stream);
int fpl_stem_conv_wgrad(const float* x, const void* dy, int dy_c8tot, int dy_c8off, float* dw,
                        int n, int cin, int d, int h, int w_, int cout, int kd, void* stream);
/* head: unet2d5_dsbn.py:293-294, nn.Conv3d(C0, classes, (1,3,3), padding (0,1,1)); logits fp32 NCDHW. */
int fpl_head_conv_fwd(const void* x, int x_c8tot, int x_c8off, const float* w, const float* bias,
                      float* logits, int n, int d, int h, int w_, int cin, int classes, void* stream);
/* The head on tcgen05: `image16` / `bias16` are the staged image / bias of the head weights zero-padded to
 * 16 output channels ((1,3,3) taps, kd = 1); the epilogue writes the first `classes` channels as fp32 NCDHW. */
int fpl_head_conv_tc(const void* x, int x_c8tot, int x_c8off, const void* image16, const float* bias16,
                     float* logits, int n, int d, int h, int w, int cin, int classes, void* stream);
/* fp32 NCDHW [N,c,D,H,W] -> C8-planar bf16 channel groups (`groups` x 8 channels, zero padded) at
 * (out_c8tot, out_c8off); chan_sum (fp32[c], may be NULL, c <= 16) ACCUMULATES the per-channel sums (the
 * head's bias gradient when x is dlogits).  Feeds dlogits / the image to the tensor-core dgrad / wgrad. */
int fpl_pack_ncdhw_to_c8(const float* x, int c, void* out, int out_c8tot, int out_c8off, int groups,
                         float* chan_sum, int n, int d, int h, int w, void* stream);
/* dlogits fp32 NCDHW -> dx C8-planar bf16; dw[classes][cin][1][3][3], db[classes] accumulated. */
int fpl_head_conv_bwd(const void* x, int x_c8tot, int x_c8off, const float* w, const float* dlogits,
                      void* dx, int dx_c8tot, int dx_c8off, float* dw, float* db,
                      int n, int d, int h, int w_, int cin, int classes, void* stream);

/* ---- (a') ConvTranspose3d k2 s2: unet2d5_dsbn.py:152,181 (w fp32 [Cin][Cout][2][2][2]) ---- */
int fpl_convt_k2s2_fwd(const void* x, int x_c8tot, int x_c8off, const float* w, const float* bias,
                       void* y, int y_c8tot, int y_c8off, int n, int d, int h, int w_, int cin, int cout,
                       int kd2, void* stream);   /* kd2 = 2 (3-D) or 1 ((1,2,2), 2.5-D levels) */
/* dy at the up-sampled resolution; dx (may be NULL) at the input resolution;
 * dw/db accumulated. */
int fpl_convt_k2s2_bwd(const void* x, int x_c8tot, int x_c8off, const float* w,
                       const void* dy, int dy_c8tot, int dy_c8off,
                       void* dx, int dx_c8tot, int dx_c8off, float* dw, float* db,
                       int n, int d, int h, int w_, int cin, int cout, int kd2, void* stream);

/* The same three operations on tcgen05 (csrc/convt_tc.cu): the stride-2 sub-lattice of one tap is fetched by TMA
 * with elementStrides = 2, fwd scatters its epilogue into (y_c8tot, y_c8off).  Images come from
 * fpl_convt_prep_weight (mode 0: forward operand, mode 1: dgrad operand); need cin % 16 == 0, cout % 16 == 0. */
int64_t fpl_convt_weight_image_bytes(int cin, int cout, int kd2);
int fpl_convt_prep_weight(const float* w, int cin, int cout, int kd2, int mode, void* image, void* stream);
int fpl_convt_prep_weight_batch(int count, const float* const* h_w, const int* h_cin, const int* h_cout,
                                const int* h_kd2, const int* h_mode, void* const* h_images, void* stream);
int fpl_convt_k2s2_fwd_tc(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias, void* y,
                          int y_c8tot, int y_c8off, int n, int d, int h, int w, int cin, int cout, int kd2, void* stream);
int fpl_convt_k2s2_dgrad_tc(const void* dy, int dy_c8tot, int dy_c8off, const void* image_t, void* dx, int dx_c8tot,
                            int dx_c8off, int n, int d, int h, int w, int cin, int cout, int kd2, void* stream);
/* dW[cin][cout][kd2][2][2] (fp32) ACCUMULATED into. */
int fpl_convt_k2s2_wgrad_tc(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                            float* dw, int n, int d, int h, int w, int cin, int cout, int kd2, void* stream);
/* Tap-major variant: scratch S[tap][cout][cin] (fp32, ACCUMULATED into); fold it into the nn.ConvTranspose3d layout
 * [cin][cout][kd2][2][2] with fpl_wgrad_tapmajor_to_dw_batch, passing the tap count NEGATED (-4*kd2). */
int fpl_convt_k2s2_wgrad_tc_tapmajor(const void* x, int x_c8tot, int x_c8off, const void* dy, int dy_c8tot, int dy_c8off,
                                     float* scratch, int n, int d, int h, int w, int cin, int cout, int kd2, void* stream);

/* ---- (b) DSBN BatchNorm3d + PReLU + Dropout + MaxPool: net_run_dsbn/dsbn.py:54-57,
 *          unet2d5_dsbn.py:76-81,104-106 ---- */

/* stats(double[2C]) -> scale/shift (fp32[C]) and save_mean/save_invstd (fp32[C]).
 * training!=0: batch statistics; running_mean/var updated with momentum (unbiased
 * var), num_batches_tracked (int64) += 1 -- pass the SELECTED domain's buffers.
 * training==0: scale/shift from the running statistics; stats unused. */
int fpl_dsbn_finalize(const double* stats, int64_t count, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, int64_t* num_batches_tracked,
                      float momentum, float eps, int training,
                      float* scale, float* shift, float* save_mean, float* save_invstd, int c, void* stream);
/* a = dropout(prelu(y*scale+shift)); optional fused 2x2x2 (pool_kd=2) or 1x2x2
 * (pool_kd=1) max-pool writing `pooled` and the argmax code `pool_idx` (uint8).
 * Dropout: p in [0,1); mask (uint8 keep flags, same C8-planar element order as a
 * dense [N][D][C/8][H][W][8] tensor) if non-NULL, else Philox4x32-10(seed + *seed_dev, offset);
 * seed_dev (device uint64, may be NULL) lets a captured CUDA graph draw a fresh mask per replay. */
int fpl_dsbn_act_fwd(const void* y, const float* scale, const float* shift, const float* slope,
                     void* a, int a_c8tot, int a_c8off,
                     void* pooled, int p_c8tot, int p_c8off, uint8_t* pool_idx, int pool_kd,
                     float drop_p, const uint8_t* drop_mask, uint64_t seed, uint64_t offset, const uint64_t* seed_dev,
                     int n, int d, int h, int w, int c, void* stream);
/* fpl_dsbn_finalize fused into the prologue of fpl_dsbn_act_fwd (one launch per layer instead of two):
 * every block derives the affine map of its 8 channels from `stats`, one block per channel group
 * publishes scale/shift/save_mean/save_invstd and updates the running statistics. */
int fpl_dsbn_bn_act_fwd(const void* y, const double* stats, int64_t count, const float* gamma, const float* beta,
                        float* running_mean, float* running_var, int64_t* num_batches_tracked, float momentum,
                        float eps, int training, float* scale, float* shift, float* save_mean, float* save_invstd,
                        const float* slope, void* a, int a_c8tot, int a_c8off, void* pooled, int p_c8tot, int p_c8off,
                        uint8_t* pool_idx, int pool_kd, float drop_p, const uint8_t* drop_mask, uint64_t seed,
                        uint64_t offset, const uint64_t* seed_dev, int n, int d, int h, int w, int c, void* stream);
/* Backward.  Gradient wrt the activated output = g1 (C8-planar slice, may be NULL)
 * + max-pool scatter of g_pool through pool_idx (may be NULL).  With dz the gradient
 * wrt the BN output and xhat = (y-mean)*invstd:
 *   pass 1 (reduce) ACCUMULATES red = double[2C+1] {sum dz [C], sum dz*xhat [C], dslope};
 *   pass 2 (apply) writes dy (bf16, dense C8-planar) = scale*(dz - mean(dz) - xhat*mean(dz*xhat))
 *                  (training) or scale*dz (training==0, BN is a fixed affine map);
 *   finalize ACCUMULATES dgamma/dbeta/dslope/dbias_conv (fp32; any may be NULL) from red.
 * The dropout mask is regenerated from (seed, offset) or read from drop_mask. */
int fpl_dsbn_act_bwd_reduce(const void* y, const void* g1, int g1_c8tot, int g1_c8off,
                            const void* g_pool, int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                            const float* scale, const float* shift, const float* save_mean,
                            const float* save_invstd, const float* slope,
                            float drop_p, const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                            const uint64_t* seed_dev, double* red, int n, int d, int h, int w, int c, void* stream);
int fpl_dsbn_act_bwd_apply(const void* y, const void* g1, int g1_c8tot, int g1_c8off,
                           const void* g_pool, int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                           const float* scale, const float* shift, const float* save_mean,
                           const float* save_invstd, const float* slope,
                           float drop_p, const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                           const uint64_t* seed_dev, const double* red, int training, void* dy,
                           int n, int d, int h, int w, int c, void* stream);
/* fpl_dsbn_act_bwd_apply with fpl_dsbn_bwd_finalize fused in (same accumulate semantics, any pointer may be NULL). */
int fpl_dsbn_act_bwd_apply_fin(const void* y, const void* g1, int g1_c8tot, int g1_c8off,
                               const void* g_pool, int gp_c8tot, int gp_c8off, const uint8_t* pool_idx, int pool_kd,
                               const float* scale, const float* shift, const float* save_mean,
                               const float* save_invstd, const float* slope,
                               float drop_p, const uint8_t* drop_mask, uint64_t seed, uint64_t offset,
                               const uint64_t* seed_dev, const double* red, int training, void* dy,
                               int n, int d, int h, int w, int c, void* stream,
                               float* dgamma, float* dbeta, float* dslope, float* dbias_conv);
int fpl_dsbn_bwd_finalize(const double* red, const float* scale, const float* save_invstd, int training,
                          float* dgamma, float* dbeta, float* dslope, float* dbias_conv, int c, void* stream);

/* ---- (d) pixel/image-weighted Dice + CE: loss/seg/dice.py:20-57, ce.py:23-44, util.py:85-107 ---- */

/* sums = double[6C+3]: I_c, Y_c, P_c, sum_w, sum_w_ce, then the hard-Dice counters of agent_seg.py:472-476
 * (sum onehot(argmax)*y, sum y, sum onehot(argmax)), then sum_{c,v} p*log2(p + 1e-10) (only filled by the _ex form with
 * want_entropy) -- ACCUMULATED into.  logits/soft_y fp32 NCDHW, weight fp32 [N,1,D,H,W] or NULL. */
int fpl_dice_ce_reduce(const float* logits, const float* soft_y, const float* weight,
                       double* sums, int n, int c, int64_t spatial, void* stream);
/* loss (fp32[1], may be NULL) and dlogits (fp32 NCDHW, may be NULL) from the sums; dlogits =
 * grad_scale * (*grad_scale_dev if non-NULL) * d(w_dice*Dice + w_ce*CE)/dlogits, so the upstream
 * gradient of autograd can stay on the device. */
int fpl_dice_ce_grad(const float* logits, const float* soft_y, const float* weight,
                     const double* sums, float w_dice, float w_ce, float grad_scale,
                     const float* grad_scale_dev, float* loss, float* dlogits,
                     int n, int c, int64_t spatial, void* stream);
/* Device data path + entropy term (SURVEY 8 f-3, a12).  Ground truth: soft_y (fp32 [N,C,S]) or, when soft_y is NULL,
 * a uint8 label map [N,S] whose one-hot is built in the kernel (LabelToProbability, transform/label_convert.py:82-88).
 * Pixel weight: weight (fp32 [N,S]) or, when weight is NULL, a uint8 agreement code [N,S] (0/1/2 = weight 0/0.5/1 of
 * data/get_pixel_weight.py:21-26); image_weight (fp32 [N], may be NULL) is folded into the code exactly as
 * NiftyDataset.set_weight_ (io/nifty_dataset.py:165-168): w < 1 -> 0, else w * image_weight[n].  10 instead of 20
 * bytes/voxel at C = 2 in the reduce pass.  w_entropy weighs the regulariser -sum p*log2(p+1e-10)/(N*D*H*W) of
 * agent_seg.py:353,467 (value and gradient); want_entropy makes the reduce pass accumulate its sum.  prob_input != 0:
 * `logits` already hold probabilities (loss_softmax = False, loss/seg/abstract.py:16-21): no softmax, d/dp returned.
 * n_global (grad form; 0 = n): number of samples the sums cover when the caller all-reduced them over data-parallel ranks
 * between the two calls -- Dice and CE are then those of the GLOBAL batch, as nn.DataParallel computes them
 * (agent_seg.py:695, loss/seg/dice.py:29-35). */
int fpl_dice_ce_reduce_ex(const float* logits, const float* soft_y, const uint8_t* label, const float* weight,
                          const uint8_t* weight_code, const float* image_weight, double* sums, int n, int c,
                          int64_t spatial, int want_entropy, int prob_input, void* stream);
int fpl_dice_ce_grad_ex(const float* logits, const float* soft_y, const uint8_t* label, const float* weight,
                        const uint8_t* weight_code, const float* image_weight, const double* sums,
                        float w_dice, float w_ce, float w_entropy, float grad_scale, const float* grad_scale_dev,
                        float* loss, float* dlogits, int n, int c, int64_t spatial, int prob_input, int n_global,
                        void* stream);
/* Loss value only (one small launch, no gradient pass): loss[0] as fpl_dice_ce_grad_ex writes it, and -- when hard_dice
 * is not NULL -- hard_dice[c] = (2*HI_c + 1e-5) / (HY_c + HP_c + 1e-5), the class-wise Dice of the argmax one-hot
 * against the ground truth that training_all logs every iteration (agent_seg.py:472-476, loss/seg/util.py:85-107), from
 * the hard counters of the same sums (replaces five element-wise torch kernels per domain pass). */
int fpl_dice_ce_loss_ex(const float* logits, const float* soft_y, const uint8_t* label, const float* weight,
                        const uint8_t* weight_code, const float* image_weight, const double* sums,
                        float w_dice, float w_ce, float w_entropy, float* loss, double* hard_dice, int n, int c,
                        int64_t spatial, int prob_input, int n_global, void* stream);

/* ---- (c) pseudo-label filter: agent_seg.py:897-931,1045-1050; data/get_pixel_weight.py:21-26;
 *          io/nifty_dataset.py:165-168 ---- */

/* logits fp32 [B,C,spatial] -> uint8 argmax labels (first max wins). */
int fpl_argmax_label(const float* logits, uint8_t* label, int b, int c, int64_t spatial, void* stream);
/* K MC-dropout logits maps of ONE volume ([K][C][spatial], passes may live in
 * separate buffers: logits_k[k]) -> out (double[2]: sum of per-voxel population
 * variance over classes, boundary voxel count), optional uncertainty map fp32[spatial]. */
int fpl_mc_uncertainty(const float* const* h_logits_k, int k, int c, int64_t spatial,
                       double* out, float* uncertainty_map, void* stream);
/* Largest K fpl_mc_uncertainty accepts (agent_seg.py:898 hard-codes 6): the host validates
 * `fpl_mc_passes` against it BEFORE running the K forwards. */
int fpl_mc_uncertainty_max_passes(void);
/* Two logits maps (target pass, fake-source pass) -> two uint8 label maps and the
 * agreement weight 1 - 0.5*[a != b]; if fold_image_weight != 0 the weight is folded
 * as set_weight_ does: (w < 1 ? 0 : w) * image_weight.  out_count (int64[1], may be
 * NULL) accumulates the number of disagreeing voxels. */
int fpl_agree_weight(const float* logits_tgt, const float* logits_src, uint8_t* label_tgt, uint8_t* label_src,
                     float* weight, int fold_image_weight, float image_weight, long long* out_count,
                     int c, int64_t spatial, void* stream);

/* ---- (c') sliding window: net_run_dsbn/infer_func.py:96-112, 202-219 ---- */

/* out[b,c, d0+i, h0+j', w0+k'] += scale * patch[b,c,i,j,k] with j' = ph-1-j when
 * flip_h (k' likewise for flip_w); count (may be NULL) += 1 on the same voxels. */
int fpl_window_accumulate(const float* patch, float* out, float* count, int b, int c,
                          int vd, int vh, int vw, int d0, int h0, int w0, int pd, int ph, int pw,
                          int flip_h, int flip_w, float scale, void* stream);
/* out = out / count * scale (count may be NULL). */
int fpl_window_normalize(float* out, const float* count, float scale, int64_t numel, void* stream);

#ifdef __cplusplus
}
#endif
#endif

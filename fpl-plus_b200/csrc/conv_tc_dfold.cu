// Depth-folded implicit-GEMM conv3d (k 3x3x3, "same") for the SMALL-channel layers, where a tcgen05.mma
// M=128 x N=Cout x K=16 is paced by the shared-memory feed of its A operand (4 KB per instruction), not by the math:
// instead of 27 MMAs (N = Cout) per OUTPUT plane, every INPUT plane tile issues 9 MMAs whose N spans the three
// output planes it contributes to,  D[z-1 | z | z+1] += A(z) * [W_kd=2 | W_kd=1 | W_kd=0]   (N = 3*Cout),
// so the A tile is fetched from shared memory 9 times instead of 27 and from L2 once instead of three times.
//   * a CTA owns a (n, 16x8 tile, depth chunk of DC planes) column: TMEM holds DC accumulators side by side
//     (DC*Cout columns); the first / last input planes of a chunk use N = Cout or 2*Cout sub-ranges of B;
//   * all 27 taps of the layer's weights stay RESIDENT in shared memory (<= 110 KB) for the kernel's lifetime;
//   * accumulators are kept zeroed by the epilogue (tcgen05.st after each read), every MMA accumulates;
//   * output plane p is complete once input plane p+1 has been issued: its epilogue (bias, bf16 store, BatchNorm
//     partial sums) runs under the MMAs of the following planes.
// Same operands, contract and epilogue as conv3d_tc_kernel (conv_tc.cu); forward and dgrad.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/fplplus_b200.h"

namespace {

constexpr int kTileH = 16, kTileW = 8;
constexpr int kBoxH = kTileH + 2, kBoxW = kTileW + 2;
constexpr int kPlaneBytes = kBoxH * kBoxW * 16;
constexpr int kThreadsD = 192;
constexpr int kMaxStagesD = 8;
constexpr int kMaxDC = 16;

struct DfParams {
    const __nv_bfloat16* image;      // [slice][tap9][cin/16][2][3*nb][8]
    const float* bias;
    bf16x8* y;
    int y_c8tot, y_c8off;
    double* stats;
    int N, D, H, W, cin, cout;
    int x_c8tot, x_c8off;
    int nb, nslices, dc, ndc;        // dc: output planes per depth chunk; ndc = ceil(D/dc)
    int a_bytes, b_bytes, stages, tmem_cols;
    int pb;                          // input planes per TMA box (= per pipeline stage)
    int tiles_h, tiles_w, total_items;
    int full_items;                  // items [0, full_items) own dc output planes; the rest are HALF chunks (tail balance)
    int taps;                        // 9 (k 3x3x3) or 1 (k 3x1x1: only the centre in-plane tap)
    int a_ksteps;                    // distinct 16-channel K steps of A (B K step j reads A K step j % a_ksteps)
    EpiAct act;                      // act.scale != NULL: inference epilogue (affine + PReLU) instead of + bias
};

__device__ __forceinline__ void tmem_st_zero16(uint32_t taddr) {
    const uint32_t z = 0u;
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};"
        ::"r"(taddr), "r"(z) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

struct DfItem {
    int n, d0, h0, w0, slice, dcount;
};

__device__ __forceinline__ DfItem decode_item(const DfParams& P, int t) {
    DfItem c;
    // the last (items mod grid) chunks are cut into two half-depth items each, so that the CTAs that would have walked one
    // more full chunk than the others walk half a chunk more (1024 chunks on 296 CTAs: 3.5 instead of 4 chunk times)
    int half = -1;
    if (t >= P.full_items) {
        const int u = t - P.full_items;
        half = u & 1;
        t = P.full_items + (u >> 1);
    }
    int tw = t % P.tiles_w; t /= P.tiles_w;
    int th = t % P.tiles_h; t /= P.tiles_h;
    int ch = t % P.ndc; t /= P.ndc;
    c.n = t % P.N;
    c.slice = t / P.N;
    c.h0 = th * kTileH;
    c.w0 = tw * kTileW;
    c.d0 = ch * P.dc;
    c.dcount = min(P.dc, P.D - c.d0);
    if (half >= 0) {
        const int hd = P.dc / 2;
        c.d0 += half * hd;
        c.dcount = max(0, min(hd, c.dcount - half * hd));
    }
    return c;
}

// NCH = nb / 16.  For NCH == 1 (Cout 16: the full-resolution layers, where a CTA walks ~60 planes per launch; 64
// accumulator registers for Cout 32 would cost the second resident CTA) the per-channel sums of the epilogue (forward BatchNorm statistics) are
// accumulated PER THREAD (32 registers per chunk) and transposed across the warp once per CTA; the transposing
// butterfly per plane (31 shuffles + ~90 ALU instructions on warps that have an SM sub-partition to themselves) made
// the epilogue the pacing stage of the 16 -> 16 layers (52 us without statistics, 65 us with; tools/epi_probe.py).
template <int NCH>
__global__ void __launch_bounds__(kThreadsD, 2) conv3d_tc_dfold_kernel(const __grid_constant__ CUtensorMap xmap, DfParams P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    // [resident weights of this CTA's slice][A stage ring][barriers][bias]
    uint8_t* b_sm = smem;
    uint8_t* ring = smem + P.b_bytes;
    const uint32_t stage_bytes = (uint32_t)(P.pb * P.a_bytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)P.stages * stage_bytes);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + kMaxStagesD;
    uint64_t* done_bar = bars + 2 * kMaxStagesD;                  // [kMaxDC] output plane complete
    uint64_t* acc_free = bars + 2 * kMaxStagesD + kMaxDC;         // all accumulators drained and zeroed
    uint64_t* w_bar = bars + 2 * kMaxStagesD + kMaxDC + 1;        // resident weights landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStagesD + kMaxDC + 2);
    float* bias_sm = reinterpret_cast<float*>(bars + 2 * kMaxStagesD + kMaxDC + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&xmap) : "memory");
        for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int p = 0; p < kMaxDC; ++p) mbar_init(&done_bar[p], 1);
        mbar_init(acc_free, 4);
        mbar_init(w_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    FPL_PDL_WAIT();      // prologue above overlapped the previous kernel's tail; from here on its results are visible
    float* scale_sm = bias_sm + P.cout;
    const bool fuse_act = P.act.scale != nullptr;
    for (int i = threadIdx.x; i < P.cout; i += kThreadsD) {
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
            int cur_slice = -1;
            int stage = 0; uint32_t phase = 0;
            for (int t = blockIdx.x; t < P.total_items; t += gridDim.x) {
                const DfItem c = decode_item(P, t);
                if (c.dcount == 0) continue;
                if (c.slice != cur_slice) {
                    // items are ordered slice-major, so a CTA (re)loads the resident weights at most nslices times;
                    // the MMA warp has drained every earlier stage before it waits on w_bar again (see below)
                    cur_slice = c.slice;
                    mbar_expect_tx(w_bar, (uint32_t)P.b_bytes);
                    const uint8_t* src = reinterpret_cast<const uint8_t*>(P.image) + (size_t)c.slice * P.b_bytes;
                    for (int off = 0; off < P.b_bytes; off += 32768) {
                        const int nbytes = min(32768, P.b_bytes - off);
                        bulk_load(b_sm + off, src + off, (uint32_t)nbytes, w_bar);
                    }
                }
                // ONE box per stage = pb consecutive input planes (planes outside the volume: TMA zero fill).  A box costs
                // the TMA unit ~400 cycles of fixed overhead + ~8 per row per CTA whatever its size (profiles/r02c_dfold_knobs.log:
                // the load pipeline alone took 28 us of the 47 us of the 16 -> 16 layer with one 5.8 KB box per plane)
                for (int z = c.d0 - 1; z <= c.d0 + c.dcount; z += P.pb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_expect_tx(&full_bar[stage], stage_bytes);
                    tma_load_5d(ring + (size_t)stage * stage_bytes, &xmap, &full_bar[stage], (c.w0 - 1) * 8, c.h0 - 1, P.x_c8off, z, c.n);
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (warp-uniform loop, one elected lane issues) =====================
        const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | (8u << 24);
        const uint64_t a_hi = make_desc(0, kPlaneBytes, kBoxW * 16);
        const uint64_t b_hi = make_desc(0, (uint32_t)(3 * P.nb) * 16, 128);
        const uint32_t b_u = smem_u32(b_sm) >> 4, ring_u = smem_u32(ring) >> 4;
        const int ksteps = P.cin / 16;
        const uint64_t b_kstep = (uint64_t)(2 * 3 * P.nb);             // 16-byte units per 16-channel K step
        const uint64_t b_tap = (uint64_t)ksteps * b_kstep;
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        uint32_t item_phase = 0, w_phase = 0;
        int cur_slice = -1;
        for (int t = blockIdx.x; t < P.total_items; t += gridDim.x) {
            const DfItem c = decode_item(P, t);
            if (c.dcount == 0) continue;
            if (c.slice != cur_slice) {
                cur_slice = c.slice;
                mbar_wait(w_bar, w_phase);
                w_phase ^= 1;
            }
            mbar_wait(acc_free, item_phase);                            // accumulators drained + zeroed
            tc_fence_after();
            for (int r0 = -1; r0 <= c.dcount; r0 += P.pb) {             // one box = input planes z = d0 + r0 .. + pb - 1
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                for (int q = 0; q < P.pb; ++q) {
                    const int r = r0 + q, z = c.d0 + r;
                    if (r > c.dcount) break;
                    if (z >= 0 && z < P.D) {
                        // output planes r-1+j, j in [jlo, jhi], clipped to the chunk
                        const int jlo = r < 1 ? 1 - r : 0;
                        const int jhi = r > c.dcount - 2 ? c.dcount - r : 2;
                        const uint32_t ncols = (uint32_t)(jhi - jlo + 1) * (uint32_t)P.nb;
                        const uint32_t idesc = idesc0 | ((ncols >> 3) << 17);
                        const uint32_t d_tmem = tmem_base + (uint32_t)(r - 1 + jlo) * (uint32_t)P.nb;
                        const uint32_t a_base = ring_u + (((uint32_t)stage * stage_bytes + (uint32_t)(q * P.a_bytes)) >> 4);
                        const uint32_t b_base = b_u + (uint32_t)(jlo * P.nb);
                        // 64-bit adds of warp-uniform values (the 14-bit start-address field never carries): the descriptor
                        // arithmetic stays on the uniform datapath (hi | uint32 expressions cost ~10 instructions per MMA)
                        uint64_t b_j = b_hi + (uint64_t)b_base;
                        for (int j = 0; j < ksteps; ++j, b_j += b_kstep) {
                            const uint64_t a_j = a_hi + (uint64_t)(a_base + (uint32_t)(j % P.a_ksteps) * (2 * kPlaneBytes / 16));
                            if (P.taps == 1) {
                                if (leader) umma_bf16(d_tmem, a_j + (uint64_t)(kBoxW + 1), b_j, idesc, 1u);
                            } else {
                                uint64_t bdesc = b_j;
#pragma unroll
                                for (int t9 = 0; t9 < 9; ++t9, bdesc += b_tap) {
                                    const uint64_t adesc = a_j + (uint64_t)((t9 / 3) * kBoxW + (t9 % 3));
                                    if (leader) umma_bf16(d_tmem, adesc, bdesc, idesc, 1u);
                                }
                            }
                        }
                    }
                    if (r >= 1) {                                       // output plane r-1 has all its contributions
                        if (leader) umma_commit(&done_bar[r - 1]);
                        __syncwarp();
                    }
                }
                if (leader) umma_commit(&empty_bar[stage]);
                __syncwarp();
                if (++stage == P.stages) { stage = 0; phase ^= 1; }
            }
            // a short last chunk: complete the unused plane barriers too, so that every barrier flips once per item
            for (int p = c.dcount; p < P.dc; ++p) {
                if (leader) umma_commit(&done_bar[p]);
                __syncwarp();
            }
            item_phase ^= 1;
        }
        FPL_PDL_TRIGGER();   // this CTA has issued its last tile: the next kernel of the stream may be scheduled as SMs drain
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        const int hl = row / kTileW, wl = row % kTileW;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        constexpr int kMaxChunks = NCH;                                 // nb = 16 * NCH <= 64
        constexpr bool kThreadAcc = NCH <= 2;
        float run[kMaxChunks];
        float tacc[kThreadAcc ? NCH : 1][32];
#pragma unroll
        for (int k = 0; k < kMaxChunks; ++k) run[k] = 0.0f;
#pragma unroll
        for (int k = 0; k < (kThreadAcc ? NCH : 1); ++k)
#pragma unroll
            for (int i = 0; i < 32; ++i) tacc[k][i] = 0.0f;
        const bool want_stats = P.stats != nullptr;
        constexpr int nchunk16 = NCH;
        // zero every accumulator once, then hand them to the MMA warp
        for (int col = 0; col < P.dc * P.nb; col += 16) tmem_st_zero16(lane_base + (uint32_t)col);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_free);
        uint32_t item_phase = 0;
        int cur_slice = -1;
        const float act_slope = fuse_act ? __ldg(P.act.slope) : 0.0f;
        for (int t = blockIdx.x; t < P.total_items; t += gridDim.x) {
            const DfItem c = decode_item(P, t);
            if (c.dcount == 0) continue;
            if (want_stats && c.slice != cur_slice) {
                if (cur_slice >= 0) {
#pragma unroll
                    for (int k = 0; k < kMaxChunks; ++k)
                        if (k < nchunk16) {
                            if (kThreadAcc) {
                                warp_transpose_sum32(tacc[k], lane);
                                run[k] += tacc[k][0];
#pragma unroll
                                for (int i = 0; i < 32; ++i) tacc[k][i] = 0.0f;
                            }
                            atomicAdd(P.stats + (lane >> 4) * P.cout + cur_slice * P.nb + k * 16 + (lane & 15), (double)run[k]);
                            run[k] = 0.0f;
                        }
                }
                cur_slice = c.slice;
            }
            const int h = c.h0 + hl, w = c.w0 + wl;
            const bool valid = h < P.H && w < P.W;
            const int64_t HW = (int64_t)P.H * P.W;
            for (int p = 0; p < c.dcount; ++p) {
                mbar_wait(&done_bar[p], item_phase);
                tc_fence_after();
                const int64_t out_base = (((int64_t)c.n * P.D + c.d0 + p) * P.y_c8tot + P.y_c8off + (c.slice * P.nb) / 8) * HW +
                                         (int64_t)h * P.W + w;
#pragma unroll
                for (int k = 0; k < kMaxChunks; ++k) {
                    if (k < nchunk16) {
                        const int c0 = k * 16;
                        const uint32_t taddr = lane_base + (uint32_t)(p * P.nb + c0);
                        uint32_t r[16];
                        tmem_ld16(taddr, r);
                        tmem_ld_wait();
                        tmem_st_zero16(taddr);                          // leave the slot clean for the next item
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
                            // inference: eval-mode BatchNorm + PReLU applied here (no activation pass follows)
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
                        }
                        if (valid) {
                            st_bf16x8(P.y + out_base + (int64_t)(c0 / 8) * HW, v);
                            st_bf16x8(P.y + out_base + (int64_t)(c0 / 8 + 1) * HW, v + 8);
                        }
                        if (want_stats) {
                            if (kThreadAcc) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) {
                                    const float xv = valid ? v[i] : 0.0f;
                                    tacc[k][i] += xv;
                                    tacc[k][16 + i] = fmaf(xv, xv, tacc[k][16 + i]);
                                }
                            } else {
#pragma unroll
                                for (int i = 0; i < 16; ++i) {
                                    v[i] = valid ? v[i] : 0.0f;
                                    v[16 + i] = v[i] * v[i];
                                }
                                warp_transpose_sum32(v, lane);
                                run[k] += v[0];
                            }
                        }
                    }
                }
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_free);
            item_phase ^= 1;
        }
        if (kThreadAcc && cur_slice >= 0) {
#pragma unroll
            for (int k = 0; k < kMaxChunks; ++k) {
                warp_transpose_sum32(tacc[k], lane);
                run[k] += tacc[k][0];
            }
        }
        if (want_stats && cur_slice >= 0) {
#pragma unroll
            for (int k = 0; k < kMaxChunks; ++k)
                if (k < nchunk16)
                    atomicAdd(P.stats + (lane >> 4) * P.cout + cur_slice * P.nb + k * 16 + (lane & 15), (double)run[k]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
    }
}

// weights: fp32 [Cout][Cin][27] -> bf16 [slice][tap9][cin/16][2][3*nb][8]; column block jj of B feeds output plane
// z-1+jj of input plane z, i.e. depth tap kd = 2 - jj.  transpose_flip as in fpl_conv3d_prep_weight.
__global__ void dfold_prep_kernel(const float* __restrict__ w, __nv_bfloat16* image, int cin_eff, int cout_eff, int transpose_flip,
                                  int nb, int total, int taps) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int ksteps = cin_eff / 16, n3 = 3 * nb, T = 3 * taps;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int t = i;
        const int el = t % 8; t /= 8;
        const int nn = t % n3; t /= n3;
        const int k8 = t % 2; t /= 2;
        const int j = t % ksteps; t /= ksteps;
        const int t9 = t % taps;
        const int sl = t / taps;
        const int in = j * 16 + k8 * 8 + el;
        const int jj = nn / nb, out = sl * nb + nn % nb;
        const int tap = (2 - jj) * taps + t9;
        float v;
        if (!transpose_flip) v = w[((int64_t)out * cin_eff + in) * T + tap];
        else v = w[((int64_t)in * cout_eff + out) * T + (T - 1 - tap)];
        image[i] = __float2bfloat16_rn(v);
    }
}

struct DfCfg {
    int nb, nslices, dc, stages, a_bytes, b_bytes, tmem_cols, smem_bytes, ctas_per_sm, pb;
};

bool make_df_cfg(int cin, int cout, int d, DfCfg& c, int taps = 9, int cin_a = 0) {
    if (cin_a <= 0) cin_a = cin;
    if (cin % 16 || cout % 16 || cin > 64 || cin_a % 16 || cin_a > cin) return false;
    c.nb = cout <= 64 ? cout : (cout % 64 == 0 ? 64 : (cout % 32 == 0 ? 32 : 16));
    if (c.nb != 16 && c.nb != 32 && c.nb != 64) return false;
    c.nslices = cout / c.nb;
    if (c.nslices != 1) return false;          // resident weights are loaded once per CTA
    c.b_bytes = taps * cin * 3 * c.nb * 2;
    if (c.b_bytes > 112 * 1024) return false;
    c.a_bytes = (cin_a / 8) * kPlaneBytes;
    c.dc = c.nb == 16 ? 16 : 8;
    if (c.dc > d) c.dc = d;
    if (c.dc < 2) return false;
    int cols = c.dc * c.nb;
    c.tmem_cols = 32;
    while (c.tmem_cols < cols) c.tmem_cols *= 2;
    if (c.tmem_cols > 512) return false;
    // pb input planes per TMA box / pipeline stage; as many stages (2..4) as keep two CTAs per SM, else what fits one
    c.pb = c.a_bytes <= 2 * kPlaneBytes ? 3 : 2;      // measured: profiles/r02c_dfold_knobs.log
    // (ONE commit per box -- the producer waiting on the epilogue's plane barriers instead of its own empty barriers --
    //  was measured SLOWER for the Cin 16 layers: 16 -> 16 41.5 -> 46.3 us, pb 1: 47.0 -> 55.7 us; kept two barriers)
    const int fixed = c.b_bytes + 1024 + 512 + 2 * cout * (int)sizeof(float) + 16;
    c.stages = 0;
    for (int s = c.pb == 1 ? 6 : 4; s >= 2 && c.stages == 0; --s)
        if (fixed + s * c.pb * c.a_bytes <= 110 * 1024) c.stages = s;
    for (int s = 4; s >= 2 && c.stages == 0; --s)
        if (fixed + s * c.pb * c.a_bytes <= 220 * 1024) c.stages = s;
    if (c.stages == 0) return false;
    c.smem_bytes = fixed + c.stages * c.pb * c.a_bytes;
    if (c.smem_bytes > 220 * 1024) return false;
    c.ctas_per_sm = (c.smem_bytes <= 110 * 1024 && c.tmem_cols <= 256) ? 2 : 1;
    return true;
}

}  // namespace

extern "C" int64_t fpl_conv3d_dfold_image_bytes(int cin, int cout) {
    DfCfg c;
    if (!make_df_cfg(cin, cout, 16, c)) return -1;
    return (int64_t)c.nslices * c.b_bytes;
}

static int dfold_prep(const float* w, int cin, int cout, int transpose_flip, int taps, void* image, void* stream) {
    const int cin_eff = transpose_flip ? cout : cin, cout_eff = transpose_flip ? cin : cout;
    DfCfg c;
    FPL_REQUIRE(make_df_cfg(cin_eff, cout_eff, 16, c, taps), "fpl_conv3d_dfold_prep_weight: unsupported channels (%d -> %d)", cin_eff, cout_eff);
    const int total = c.nslices * c.b_bytes / 2;
    int blocks = (total + 255) / 256;
    if (blocks > FPL_NUM_SMS * 4) blocks = FPL_NUM_SMS * 4;
    fpl_launch(dfold_prep_kernel, blocks, 256, 0, (cudaStream_t)stream, w, (__nv_bfloat16*)image, cin_eff, cout_eff, transpose_flip, c.nb, total, taps);
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_conv3d_dfold_prep_weight(const float* w, int cin, int cout, int transpose_flip, void* image, void* stream) {
    return dfold_prep(w, cin, cout, transpose_flip, 9, image, stream);
}

/* k = (3,1,1): w is fp32 [Cout][Cin][3] */
extern "C" int fpl_conv3d_k311_prep_weight(const float* w, int cin, int cout, void* image, void* stream) {
    return dfold_prep(w, cin, cout, 0, 1, image, stream);
}

// all depth-folded images of a network in ONE launch (blockIdx.y = entry); host arrays of length count
namespace {
constexpr int kMaxDfBatch = 64;
struct DfPrepBatch {
    const float* w[kMaxDfBatch];
    __nv_bfloat16* image[kMaxDfBatch];
    int cin_eff[kMaxDfBatch], cout_eff[kMaxDfBatch], total[kMaxDfBatch];
    unsigned char tf[kMaxDfBatch], nb[kMaxDfBatch];
};
// one thread per (out, in) pair: 27 contiguous source floats -> 27 image positions (see prep_weight_batch_kernel)
__global__ void dfold_prep_batch_kernel(const __grid_constant__ DfPrepBatch B) {
    FPL_PDL_WAIT();      // everything below may read what earlier kernels of the stream wrote
    const int e = blockIdx.y;
    const float* __restrict__ w = B.w[e];
    __nv_bfloat16* image = B.image[e];
    const int cin_eff = B.cin_eff[e], cout_eff = B.cout_eff[e], nb = B.nb[e], tf = B.tf[e];
    const int ksteps = cin_eff / 16, n3 = 3 * nb;
    const int pairs = cin_eff * cout_eff;                 // nslices == 1: out == n
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < pairs; r += gridDim.x * blockDim.x) {
        const int el = r & 7, n = (r >> 3) % nb, jk = (r >> 3) / nb;      // jk = j * 2 + k8
        const int in = jk * 8 + el, out = n;
        const float* src = tf ? w + ((int64_t)in * cout_eff + out) * 27 : w + ((int64_t)out * cin_eff + in) * 27;
#pragma unroll
        for (int jj = 0; jj < 3; ++jj) {
#pragma unroll
            for (int t9 = 0; t9 < 9; ++t9) {
                const int tap = (2 - jj) * 9 + t9;
                const float v = __ldg(src + (tf ? 26 - tap : tap));
                image[(((int64_t)t9 * ksteps * 2 + jk) * n3 + jj * nb + n) * 8 + el] = __float2bfloat16_rn(v);
            }
        }
    }
}
}  // namespace

extern "C" int fpl_conv3d_dfold_prep_weight_batch(int count, const float* const* h_w, const int* h_cin, const int* h_cout,
                                                  const int* h_transpose_flip, void* const* h_images, void* stream) {
    FPL_REQUIRE(count >= 0 && count <= kMaxDfBatch, "fpl_conv3d_dfold_prep_weight_batch: count %d not in [0,%d]", count, kMaxDfBatch);
    if (count == 0) return 0;
    DfPrepBatch B;
    int max_total = 0;
    for (int e = 0; e < count; ++e) {
        const int tf = h_transpose_flip[e];
        const int cin_eff = tf ? h_cout[e] : h_cin[e], cout_eff = tf ? h_cin[e] : h_cout[e];
        DfCfg c;
        FPL_REQUIRE(make_df_cfg(cin_eff, cout_eff, 16, c), "fpl_conv3d_dfold_prep_weight_batch: unsupported channels (%d -> %d)", cin_eff, cout_eff);
        B.w[e] = h_w[e]; B.image[e] = (__nv_bfloat16*)h_images[e]; B.cin_eff[e] = cin_eff; B.cout_eff[e] = cout_eff;
        B.tf[e] = (unsigned char)tf; B.nb[e] = (unsigned char)c.nb; B.total[e] = c.nslices * c.b_bytes / 2;
        if (B.total[e] > max_total) max_total = B.total[e];
    }
    int bx = (max_total / 27 + 255) / 256;
    if (bx > 32) bx = 32;
    if (bx < 1) bx = 1;
    fpl_launch(dfold_prep_batch_kernel, dim3(bx, count), 256, 0, (cudaStream_t)stream, B);
    FPL_LAUNCH_CHECK();
    return 0;
}

static int dfold_launch(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias, void* y,
                        int y_c8tot, int y_c8off, double* stats, int n, int d, int h, int w, int cin, int cout, int taps,
                        int cin_a, void* stream, const EpiAct* act = nullptr) {
    if (cin_a <= 0) cin_a = cin;
    DfCfg c;
    FPL_REQUIRE(make_df_cfg(cin, cout, d, c, taps, cin_a), "fpl_conv3d_tc_dfold: unsupported shape (%d -> %d, depth %d)", cin, cout, d);
    FPL_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(image) & 15) == 0,
                "fpl_conv3d_tc_dfold: x/image must be 16-byte aligned");
    EncodeTiledFn encode = get_encode_fn();
    FPL_REQUIRE(encode != nullptr, "fpl_conv3d_tc_dfold: cuTensorMapEncodeTiled not available from the driver");
    CUtensorMap xmap;
    cuuint64_t gdim[5] = {(cuuint64_t)w * 8, (cuuint64_t)h, (cuuint64_t)x_c8tot, (cuuint64_t)d, (cuuint64_t)n};
    cuuint64_t gstride[4] = {(cuuint64_t)w * 16, (cuuint64_t)h * w * 16, (cuuint64_t)x_c8tot * h * w * 16,
                             (cuuint64_t)d * x_c8tot * h * w * 16};
    cuuint32_t box[5] = {(cuuint32_t)kBoxW * 8, (cuuint32_t)kBoxH, (cuuint32_t)(cin_a / 8), (cuuint32_t)c.pb, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&xmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FPL_REQUIRE(r == CUDA_SUCCESS, "fpl_conv3d_tc_dfold: cuTensorMapEncodeTiled failed (%d)", (int)r);
    DfParams P;
    P.image = (const __nv_bfloat16*)image; P.bias = bias; P.y = (bf16x8*)y; P.y_c8tot = y_c8tot; P.y_c8off = y_c8off;
    P.stats = stats; P.N = n; P.D = d; P.H = h; P.W = w; P.cin = cin; P.cout = cout;
    P.x_c8tot = x_c8tot; P.x_c8off = x_c8off;
    P.nb = c.nb; P.nslices = c.nslices; P.dc = c.dc; P.ndc = (d + c.dc - 1) / c.dc;
    P.a_bytes = c.a_bytes; P.b_bytes = c.b_bytes; P.stages = c.stages; P.tmem_cols = c.tmem_cols; P.pb = c.pb;
    P.tiles_h = (h + kTileH - 1) / kTileH; P.tiles_w = (w + kTileW - 1) / kTileW;
    int64_t total = (int64_t)P.tiles_h * P.tiles_w * P.ndc * n * c.nslices;
    FPL_REQUIRE(total < (1ll << 29), "fpl_conv3d_tc_dfold: too many items");
    int grid = FPL_NUM_SMS * c.ctas_per_sm;
    if (grid > total) grid = (int)total;
    // tail balance: when the chunks do not divide over the CTAs, the last (chunks mod grid) chunks become two half-depth
    // items each if both halves still fit one extra round (see decode_item); single-slice layers only
    P.full_items = (int)total;
    const int rem = (int)(total % grid);
    if (rem > 0 && 2 * rem <= grid && c.dc >= 8 && c.dc % 2 == 0 && d % c.dc == 0 && c.nslices == 1) P.full_items = (int)total - rem;
    P.total_items = P.full_items + 2 * ((int)total - P.full_items);
    P.taps = taps; P.a_ksteps = cin_a / 16;
    if (act != nullptr) P.act = *act; else { P.act.scale = nullptr; P.act.shift = nullptr; P.act.slope = nullptr; P.act.drop_p = 0.0f; P.act.seed = P.act.offset = 0; P.act.seed_dev = nullptr; }
    if (c.nb == 16) {
        FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_tc_dfold_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.smem_bytes));
        fpl_launch(conv3d_tc_dfold_kernel<1>, grid, kThreadsD, c.smem_bytes, (cudaStream_t)stream, xmap, P);
    } else if (c.nb == 32) {
        FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_tc_dfold_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.smem_bytes));
        fpl_launch(conv3d_tc_dfold_kernel<2>, grid, kThreadsD, c.smem_bytes, (cudaStream_t)stream, xmap, P);
    } else {
        FPL_CHECK_CUDA(cudaFuncSetAttribute(conv3d_tc_dfold_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, c.smem_bytes));
        fpl_launch(conv3d_tc_dfold_kernel<4>, grid, kThreadsD, c.smem_bytes, (cudaStream_t)stream, xmap, P);
    }
    FPL_LAUNCH_CHECK();
    return 0;
}

extern "C" int fpl_conv3d_tc_dfold(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias, void* y,
                                   int y_c8tot, int y_c8off, double* stats, int n, int d, int h, int w, int cin, int cout,
                                   void* stream) {
    return dfold_launch(x, x_c8tot, x_c8off, image, bias, y, y_c8tot, y_c8off, stats, n, d, h, w, cin, cout, 9, 0, stream);
}

/* k = (3,1,1) "same" conv (depth taps only) with the same machinery: 1 MMA (N = 3*Cout) per input plane and K step.
 * Used for the stem after fpl_patch9_c8 has turned the 9 in-plane neighbours of the 1-channel image into channels. */
extern "C" int fpl_conv3d_tc_k311(const void* x, int x_c8tot, int x_c8off, const void* image, const float* bias, void* y,
                                  int y_c8tot, int y_c8off, double* stats, int n, int d, int h, int w, int cin, int cout,
                                  int a_channels, void* stream) {
    return dfold_launch(x, x_c8tot, x_c8off, image, bias, y, y_c8tot, y_c8off, stats, n, d, h, w, cin, cout, 1, a_channels,
                        stream);
}

/* Inference forms (see fpl_conv3d_tc_act): a = prelu(acc * scale + shift) written instead of y; no dropout here (the
 * levels these kernels serve have p = 0 in every shipped configuration; callers with p > 0 use the two-kernel path). */
extern "C" int fpl_conv3d_tc_dfold_act(const void* x, int x_c8tot, int x_c8off, const void* image, void* a, int a_c8tot,
                                       int a_c8off, int n, int d, int h, int w, int cin, int cout, const float* scale,
                                       const float* shift, const float* slope, void* stream) {
    FPL_REQUIRE(scale != nullptr && shift != nullptr && slope != nullptr, "fpl_conv3d_tc_dfold_act: scale/shift/slope required");
    EpiAct act;
    act.scale = scale; act.shift = shift; act.slope = slope; act.drop_p = 0.0f; act.seed = act.offset = 0; act.seed_dev = nullptr;
    return dfold_launch(x, x_c8tot, x_c8off, image, nullptr, a, a_c8tot, a_c8off, nullptr, n, d, h, w, cin, cout, 9, 0, stream, &act);
}

extern "C" int fpl_conv3d_tc_k311_act(const void* x, int x_c8tot, int x_c8off, const void* image, void* a, int a_c8tot,
                                      int a_c8off, int n, int d, int h, int w, int cin, int cout, int a_channels,
                                      const float* scale, const float* shift, const float* slope, void* stream) {
    FPL_REQUIRE(scale != nullptr && shift != nullptr && slope != nullptr, "fpl_conv3d_tc_k311_act: scale/shift/slope required");
    EpiAct act;
    act.scale = scale; act.shift = shift; act.slope = slope; act.drop_p = 0.0f; act.seed = act.offset = 0; act.seed_dev = nullptr;
    return dfold_launch(x, x_c8tot, x_c8off, image, nullptr, a, a_c8tot, a_c8off, nullptr, n, d, h, w, cin, cout, 1, a_channels,
                        stream, &act);
}

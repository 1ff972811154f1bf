// Shared helpers for the fplplus_b200 kernels (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

// SMs the persistent / one-CTA-per-SM kernels size their grids for.  148 on a B200; a data-parallel run lowers it by the
// CTAs the NCCL all-reduce kernels hold while they overlap backward (fpl_set_sm_budget): a statically tiled 148-CTA grid
// that finds 8 SMs occupied runs its last 8 CTAs as a second wave, i.e. takes twice as long.
extern int g_fpl_num_sms;
#define FPL_NUM_SMS g_fpl_num_sms

void fpl_set_error(const char* fmt, ...);

#define FPL_CHECK_CUDA(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            fpl_set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,           \
                          cudaGetErrorString(_e));                                        \
            return 1;                                                                     \
        }                                                                                 \
    } while (0)

#define FPL_REQUIRE(cond, ...)                                                            \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            fpl_set_error(__VA_ARGS__);                                                   \
            return 2;                                                                     \
        }                                                                                 \
    } while (0)

// every kernel launch of the library goes through this macro: it bumps the launch counter that
// fpl_launch_count() reports (bench.py's "gpu_launches") and surfaces launch errors
extern unsigned long long g_fpl_launches;
#define FPL_LAUNCH_CHECK()                                                                \
    do {                                                                                  \
        __atomic_fetch_add(&g_fpl_launches, 1ull, __ATOMIC_RELAXED);                      \
        FPL_CHECK_CUDA(cudaGetLastError());                                               \
    } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------------------
// Every kernel of the library is launched with cudaLaunchAttributeProgrammaticStreamSerialization (fpl_launch): the next
// kernel of the stream may be SCHEDULED while this one is still running -- its CTAs run their prologue (barrier init,
// TMEM allocation, tensor-map prefetch, index math) and then block in griddepcontrol.wait until the whole previous grid
// has completed and flushed its memory.  ~320 dependent launches per train step otherwise pay the full
// drain-then-launch latency each, also inside a CUDA graph (the edges are captured as programmatic dependencies).
// Rules: (1) every kernel executes FPL_PDL_WAIT() before its first global read / write of data another kernel of the
// stream touches (the waits chain, so completion is transitive); (2) FPL_PDL_TRIGGER() lets the dependents be
// scheduled once every CTA of this grid has executed it (or exited).  Both are no-ops for a normally launched kernel.
#define FPL_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#define FPL_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")

extern int g_fpl_pdl;     // 1 (default) / 0: FPL_PDL environment variable, read once (api.cu)

template <typename... KArgs, typename... Args>
inline cudaError_t fpl_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_fpl_pdl;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- 16-byte bf16x8 vectors ----------------------------------------------------------
struct __align__(16) bf16x8 {
    __nv_bfloat162 v[4];
};

__device__ __forceinline__ void bf16x8_to_float(const bf16x8& a, float* f) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 t = __bfloat1622float2(a.v[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}

__device__ __forceinline__ bf16x8 float_to_bf16x8(const float* f) {
    bf16x8 r;
#pragma unroll
    for (int i = 0; i < 4; ++i) r.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return r;
}

// one 128-bit store of 8 floats rounded to bf16 (the struct assignment above compiles to four
// 32-bit stores; the epilogues and streaming kernels want a single STG.128)
__device__ __forceinline__ void st_bf16x8(void* p, const float* f) {
    __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]);
    __nv_bfloat162 c = __floats2bfloat162_rn(f[4], f[5]), d = __floats2bfloat162_rn(f[6], f[7]);
    uint4 v = make_uint4(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b),
                         *reinterpret_cast<uint32_t*>(&c), *reinterpret_cast<uint32_t*>(&d));
    *reinterpret_cast<uint4*>(p) = v;
}

// Transposing butterfly: every lane enters with 32 values w[0..31] (static indexing); on return
// lane L holds in w[0] the sum over the 32 lanes of w[L].  31 shuffles instead of 32 x 5.
__device__ __forceinline__ void warp_transpose_sum32(float* w, int lane) {
#pragma unroll
    for (int half = 16; half >= 1; half >>= 1) {
        const bool upper = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            float send = upper ? w[i] : w[i + half];
            float keep = upper ? w[i + half] : w[i];
            w[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
}

__device__ __forceinline__ bf16x8 ldg_bf16x8(const void* p) {
    int4 t = __ldg(reinterpret_cast<const int4*>(p));
    return *reinterpret_cast<bf16x8*>(&t);
}

// streaming (read-once) 16-byte load / store: keep L1 for data with reuse
__device__ __forceinline__ int4 ld_stream16(const void* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ld_stream_f4(const void* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

// C8-planar addressing: element-vector index of (n,d,c8,h,w) in a buffer with c8tot groups
__device__ __forceinline__ int64_t c8_index(int n, int d, int c8, int h, int w, int D, int C8tot, int H, int W) {
    return ((((int64_t)n * D + d) * C8tot + c8) * H + h) * (int64_t)W + w;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- Philox4x32-10 (counter based; the same stream is regenerated in backward) ------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}

// keep-mask bits for the 8 channels of element-vector `vec_index` (dense C8-planar order)
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t seed, uint64_t offset, uint64_t vec_index, float p) {
    uint64_t c = vec_index * 2 + offset;
    uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    uint4 a = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), 0u, 0u), key);
    uint4 b = philox4x32_10(make_uint4((uint32_t)(c + 1), (uint32_t)((c + 1) >> 32), 0u, 0u), key);
    uint32_t r[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float u = (float)(r[i] >> 8) * (1.0f / 16777216.0f);  // [0,1)
        bits |= (u >= p ? 1u : 0u) << i;
    }
    return bits;
}

// ---- inference epilogue of the conv kernels (BatchNorm in eval mode folded into the conv) -------------------------
// a = dropout(prelu(acc * scale + shift)):  scale = gamma / sqrt(running_var + eps),
// shift = beta + (conv bias - running_mean) * scale  (fpl_dsbn_eval_affine_batch).  scale == NULL: plain "+ bias".
struct EpiAct {
    const float* scale;
    const float* shift;
    const float* slope;
    float drop_p;
    uint64_t seed, offset;
    const unsigned long long* seed_dev;
};

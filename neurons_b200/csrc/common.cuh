// Shared host/device helpers for libneurons_mm.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>

#include "../../include/neurons_mm.h"

namespace nmm {

typedef __nv_bfloat16 bf16;

// ---- error reporting (thread-local text behind nmm_last_error) ---------------------------------
std::string &last_error_ref();
int fail(int status, const char *fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define NMM_CUDA_OK(expr)                                                                           \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            return ::nmm::fail(NMM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                               __FILE__, __LINE__);                                                 \
    } while (0)

// ---- run-time options (nmm_option; api.cu): one relaxed atomic load, initialised once from the environment ----
int64_t opt(int option);

// ---- optional per-kernel device timing (bench.py roofline): CUDA events around every launch, on the launch stream ----
enum KernelId { K_GN_STATS = 0, K_GN_TOKENS, K_LAYERNORM, K_ATTENTION, K_LINEAR_SIMT, K_LINEAR_TC, K_PACK, K_FUSED_MODULE, K_SPATIAL_ATTN, K_COUNT };
struct ProfScope {          // records start on construction, stop on destruction; no-op unless profiling is enabled
    int slot;
    cudaStream_t st;
    ProfScope(int kid, cudaStream_t stream, double flops, double bytes);
    ~ProfScope();
};

// cudaFuncSetAttribute is per device: a "done" flag per (kernel instantiation, device ordinal).  Usage:
//     static DeviceOnce once;  NMM_CUDA_OK(once.max_smem(kern, bytes));
// The flag is published only AFTER the attribute call has returned (and the call itself is serialised), so a second host
// thread on the same device can never launch a > 48 KB kernel before the attribute is in place.
struct DeviceOnce {
    std::mutex mu;
    std::atomic<bool> done[64];
    DeviceOnce() { for (auto &d : done) d.store(false, std::memory_order_relaxed); }
    template <typename K>
    cudaError_t max_smem(K kern, int bytes) {
        int dev = 0;
        const bool known = cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64;
        if (known && done[dev].load(std::memory_order_acquire)) return cudaSuccess;
        std::lock_guard<std::mutex> lk(mu);
        if (known && done[dev].load(std::memory_order_relaxed)) return cudaSuccess;
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e == cudaSuccess && known) done[dev].store(true, std::memory_order_release);
        return e;
    }
};

// Count + check a kernel launch without synchronising (stays graph-capturable).
#define NMM_LAUNCHED(name)                                                                          \
    do {                                                                                            \
        ::nmm::g_launches.fetch_add(1, std::memory_order_relaxed);                                  \
        cudaError_t _e = cudaGetLastError();                                                        \
        if (_e != cudaSuccess)                                                                      \
            return ::nmm::fail(NMM_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(_e)); \
    } while (0)

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------------------
// Every kernel of the library is launched with cudaLaunchAttributeProgrammaticStreamSerialization and starts with
// pdl_wait() (griddepcontrol.wait: the previous kernel in the stream has completed and its writes are visible) followed by
// pdl_launch_dependents(): the NEXT kernel's launch processing, CTA scheduling and data-independent prologue (barrier init,
// TMEM allocation, tensor-map prefetch) then overlap this kernel's execution instead of adding a launch bubble per kernel
// (~300 launches per UNet step).  Without the launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline bool aligned(const void *p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

// ---- geometry derived from nmm_shape -------------------------------------------------------------
struct Geo {
    int B, C, F, H, W, P, heads, dh, layers, A, max_len;
    int64_t N;       // tokens
    bool pos_enc;
    int dtype;
    bool ln_fold;    // bf16 mode with the LayerNorms folded into the QKV / GEGLU GEMMs
};
inline Geo geo_of(const nmm_shape *s) {
    Geo g;
    g.B = s->batch; g.C = s->channels; g.F = s->frames; g.H = s->height; g.W = s->width;
    g.P = s->height * s->width; g.heads = s->heads; g.dh = s->heads > 0 ? s->channels / s->heads : 0;
    g.layers = s->layers; g.A = s->attn_blocks; g.max_len = s->max_len;
    g.N = (int64_t)s->batch * s->frames * g.P; g.pos_enc = s->pos_enc != 0; g.dtype = s->dtype;
    g.ln_fold = s->ln_fold != 0 && s->dtype == NMM_BF16;
    return g;
}
inline size_t dtype_size(int dtype) { return dtype == NMM_BF16 ? 2 : 4; }      // NMM_F32, NMM_F32X3 and NMM_F32X6 store fp32
// bf16 planes of a tensor-core GEMM operand (NMM_F32X3: hi | lo, NMM_F32X6: hi | mid | lo) and the operand's bytes per element
inline int planes_of(int dtype) { return dtype == NMM_F32X3 ? 2 : dtype == NMM_F32X6 ? 3 : 1; }
inline size_t operand_size(int dtype) { return dtype == NMM_F32X6 ? 6 : dtype_size(dtype); }

// ---- device helpers ------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// Element-wise sum of N values over a group of G consecutive lanes (G a power of two, N >= G) by recursive halving: each step a lane
// keeps one half of its values and adds the partner's copy of that half (N - N/G shuffles instead of N log2 G).  Afterwards lane l of
// the group holds the N / G group totals of indices l * N/G ... in v[0 .. N/G).
template <int N, int G>
__device__ __forceinline__ void lane_group_reduce_scatter(float (&v)[N], int lane) {
#pragma unroll
    for (int o = G / 2, n = N / 2; o > 0; o >>= 1, n >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < n; i++) {
            const float send = up ? v[i] : v[i + n], keep = up ? v[i + n] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
}
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);   // .x = lo (low 16 bits), .y = hi
    return *reinterpret_cast<uint32_t *>(&t);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
// NMM_F32X3 operand format: an fp32 value as two bf16 terms, v = hi + lo + O(2^-17 |v|).  A [rows, K] fp32 operand is stored as a bf16
// [rows, 2K] tensor: row r = hi plane (K values) | lo plane (K values).  split4_store writes four consecutive values of one row.
__device__ __forceinline__ void split_bf16x2(float x, float y, uint32_t &hi, uint32_t &lo) {
    hi = pack_bf16x2(x, y);
    lo = pack_bf16x2(x - bf16_lo(hi), y - bf16_hi(hi));
}
// NMM_F32X6 operand format: three bf16 terms, hi = bf16(v), mid = bf16(v - hi), lo = bf16(v - hi - mid) (both differences exact in fp32),
// v = hi + mid + lo + O(2^-24 |v|).  A [rows, K] operand is a bf16 [rows, 3K] tensor: row r = hi plane | mid plane | lo plane.
__device__ __forceinline__ void split3_bf16x2(float x, float y, uint32_t &hi, uint32_t &mid, uint32_t &lo) {
    hi = pack_bf16x2(x, y);
    const float rx = x - bf16_lo(hi), ry = y - bf16_hi(hi);
    mid = pack_bf16x2(rx, ry);
    lo = pack_bf16x2(rx - bf16_lo(mid), ry - bf16_hi(mid));
}
// PL = 2 (NMM_F32X3) or 3 (NMM_F32X6) planes of K values per row
template <int PL = 2>
__device__ __forceinline__ void split4_store(bf16 *row, int K, int c, float a, float b, float cc, float d) {      // c % 4 == 0, row 8-byte aligned, K % 4 == 0
    if constexpr (PL == 3) {
        uint32_t h0, m0, l0, h1, m1, l1;
        split3_bf16x2(a, b, h0, m0, l0);
        split3_bf16x2(cc, d, h1, m1, l1);
        *reinterpret_cast<uint2 *>(row + c) = make_uint2(h0, h1);
        *reinterpret_cast<uint2 *>(row + K + c) = make_uint2(m0, m1);
        *reinterpret_cast<uint2 *>(row + 2 * K + c) = make_uint2(l0, l1);
    } else {
        uint32_t h0, l0, h1, l1;
        split_bf16x2(a, b, h0, l0);
        split_bf16x2(cc, d, h1, l1);
        *reinterpret_cast<uint2 *>(row + c) = make_uint2(h0, h1);
        *reinterpret_cast<uint2 *>(row + K + c) = make_uint2(l0, l1);
    }
}
template <int PL = 2>
__device__ __forceinline__ void split1_store(bf16 *row, int K, int c, float v) {
    const bf16 h = __float2bfloat16_rn(v);
    row[c] = h;
    const float r = v - __bfloat162float(h);
    const bf16 m = __float2bfloat16_rn(r);
    row[K + c] = m;
    if constexpr (PL == 3) row[2 * K + c] = __float2bfloat16_rn(r - __bfloat162float(m));
}

// exact (erf) GELU, as torch.nn.functional.gelu default -- motion_module_new.py:510-518
__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }
// Same function from Abramowitz-Stegun 7.1.28, erfc(x) = (1 + a1 x + ... + a6 x^6)^-16 for x >= 0 (|error| <= 3e-7), written as
//   GELU(v) = v * Phi(v),  Phi(v) = 1 - r/2 (v >= 0),  r/2 (v < 0),  r = erfc(|v| / sqrt 2)
// branch-free, 13 instructions with ONE SFU op (the approximate reciprocal).  Used by the bf16 GEGLU epilogue, which is
// instruction-issue bound at K = 320 (128 x 128 GELUs per tile against 2560 MMA cycles); SFU-heavier forms (logistic of a
// polynomial: ex2 + rcp, measured 1.7x slower) and SFU-free polynomials (2e-4 error at degree 13) both lose on B200.
// For |v| > ~15 the 16th power overflows to +inf and rcp gives exactly 0, i.e. Phi = 1 or 0 as it should.
__device__ __forceinline__ float gelu_erf_fast(float v) {
    // p = 2^(1/16) * (1 + a1 x + ... + a6 x^6) with x = |v| / sqrt 2 folded into the coefficients, so p^16 = 2 / erfc(x) and
    // GELU(v) = max(v, 0) - |v| * erfc(x) / 2 = max(v, 0) - |v| / p^16:  6 FFMA + 4 FMUL + 1 SFU + FMNMX + FFMA = 13 instructions
    const float a = fabsf(v);
    float p = fmaf(5.6212996640e-06f, a, 5.1055209009e-05f);
    p = fmaf(p, a, 3.9686137011e-05f);
    p = fmaf(p, a, 3.4227392389e-03f);
    p = fmaf(p, a, 2.2076998457e-02f);
    p = fmaf(p, a, 5.2075163037e-02f);
    p = fmaf(p, a, 1.0442737824e+00f);
    p = p * p; p = p * p; p = p * p; p = p * p;          // ^16
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));
    return fmaf(-a, r, fmaxf(v, 0.f));
}

// Two GELUs at once on the packed fp32x2 pipe of sm_100 (FFMA2 / FMUL2: one instruction, two fp32 lanes).  Same arithmetic per
// lane as gelu_erf_fast; the issue-bound GEGLU epilogue spends ~40 % fewer instructions per output pair.
__device__ __forceinline__ uint64_t f32x2_pack(float lo, float hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void f32x2_unpack(uint64_t v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f32x2_fma(uint64_t a, uint64_t b, uint64_t c) { uint64_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ uint64_t f32x2_mul(uint64_t a, uint64_t b) { uint64_t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ uint64_t f32x2_add(uint64_t a, uint64_t b) { uint64_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// (y0, y1) = (v0 * GELU(g0), v1 * GELU(g1))
__device__ __forceinline__ void geglu_pair(float v0, float g0, float v1, float g1, float &y0, float &y1) {
    const uint64_t a = f32x2_pack(fabsf(g0), fabsf(g1));
    uint64_t p = f32x2_fma(f32x2_pack(5.6212996640e-06f, 5.6212996640e-06f), a, f32x2_pack(5.1055209009e-05f, 5.1055209009e-05f));
    p = f32x2_fma(p, a, f32x2_pack(3.9686137011e-05f, 3.9686137011e-05f));
    p = f32x2_fma(p, a, f32x2_pack(3.4227392389e-03f, 3.4227392389e-03f));
    p = f32x2_fma(p, a, f32x2_pack(2.2076998457e-02f, 2.2076998457e-02f));
    p = f32x2_fma(p, a, f32x2_pack(5.2075163037e-02f, 5.2075163037e-02f));
    p = f32x2_fma(p, a, f32x2_pack(1.0442737824e+00f, 1.0442737824e+00f));
    p = f32x2_mul(p, p); p = f32x2_mul(p, p); p = f32x2_mul(p, p); p = f32x2_mul(p, p);
    float p0, p1, r0, r1;
    f32x2_unpack(p, p0, p1);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(p0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(p1));
    // GELU = max(g, 0) - |g| * r;  times the value
    const uint64_t gel = f32x2_fma(f32x2_pack(-fabsf(g0), -fabsf(g1)), f32x2_pack(r0, r1), f32x2_pack(fmaxf(g0, 0.f), fmaxf(g1, 0.f)));
    f32x2_unpack(f32x2_mul(f32x2_pack(v0, v1), gel), y0, y1);
}

// ---- internal kernels' host launchers (defined in the .cu files) ----------------------------------
// GroupNorm
size_t gn_partial_bytes(const Geo &g);
int gn_splits_of(const Geo &g);          // partial (sum, sumsq) pairs per (b, f, group) written by gn_stats
// mean / rstd of one (b, f, group) from the partial sums of gn_stats (fp64 accumulation; biased variance, as torch.nn.GroupNorm)
__device__ __forceinline__ void gn_finalize_one(const double *__restrict__ partial, int bf_grp, int splits, double count, float eps,
                                                float &mean, float &rstd) {
    double a = 0, c2 = 0;
    for (int i = 0; i < splits; i++) {
        a += partial[((int64_t)bf_grp * splits + i) * 2 + 0];
        c2 += partial[((int64_t)bf_grp * splits + i) * 2 + 1];
    }
    double m = a / count;
    double var = c2 / count - m * m;
    if (var < 0) var = 0;
    mean = (float)m;
    rstd = (float)(1.0 / sqrt(var + (double)eps));
}
int launch_gn_stats(const Geo &g, const nmm_shape *s, const void *x, double *partial, cudaStream_t st);
// splits_override > 0: `partial` holds that many (sum, sum of squares) pairs per (b, f, group) instead of gn_splits_of(g) -- 1 for
// caller-provided "sums" (precomputed statistics, SURVEY 8(f) N1)
int launch_gn_finalize(const Geo &g, const nmm_shape *s, const double *partial, float *mean, float *rstd, cudaStream_t st, int splits_override = 0);
int launch_y_sums_tiles(const float2 *part, double *sums, int B, int F, int tiles_per_b, cudaStream_t st);
int launch_y_sums_channels(const float2 *part, double *sums, int BF, int C, int P, cudaStream_t st);
int launch_gn_partial_to_sums(const Geo &g, const double *partial, double *sums, cudaStream_t st);
int launch_gn_tokens(const Geo &g, const nmm_shape *s, const Geo &full, const void *x, const double *partial, const float *gn_w,
                     const float *gn_b, void *tokens, cudaStream_t st, int splits_override = 0);      // NMM_F32X3 / X6: tokens = bf16 [N, 2C / 3C] planes
// LayerNorm (+PE)
int launch_layernorm_pe(const Geo &g, const nmm_shape *s, const float *h, const float *w, const float *b,
                        const float *pe, void *out, cudaStream_t st);
// attention
int launch_temporal_attention(const Geo &g, const void *qkv, void *ctx, cudaStream_t st);

// spatial (long-sequence, flash-style) attention of the UNet's Transformer3DModel blocks: spatial_attention.cu (SURVEY 8(f) N3)
struct FlashArgs {
    const void *q, *k, *v;   // rows of heads * dh channels (a column slice of a projection output); head h = columns [h * dh, (h + 1) * dh)
    void *o;
    int64_t q_rs, kv_rs, o_rs;      // row strides (elements)
    int64_t q_bs, kv_bs, o_bs;      // image strides (elements); the k / v image of q image i is i / kv_div
    int64_t q_lo_off, kv_lo_off;    // launch_spatial_attention_x3 / _x6 only: element offset from one bf16 plane to the next inside a q / k-v row
    int Lq, Lkv, heads, images, kv_div, dh;
    int dtype;                      // NMM_BF16 (mma.sync flash kernel) or NMM_F32 (fp32 kernels: tiled FMA-pipe flash or checker)
    float scale, scale_log2e;       // dh^-1/2 and dh^-1/2 * log2(e)
};
int launch_spatial_attention(const FlashArgs &a, cudaStream_t st);
bool spatial_attention_tc_eligible(const FlashArgs &a);                            // spatial_attention_tc.cu (tcgen05 / TMEM / TMA)
int launch_spatial_attention_tc(const FlashArgs &a, int variant, cudaStream_t st);
int launch_spatial_attention_x3(const FlashArgs &a, cudaStream_t st);               // spatial_attention_x3.cu: fp32-grade (hi | lo bf16 planes in, fp32 out)
int launch_spatial_attention_x6(const FlashArgs &a, cudaStream_t st);               // spatial_attention_x6.cu: fp32-exact (hi | mid | lo bf16 planes in, fp32 out)
bool spatial_attention_f32_tiled_eligible(const FlashArgs &a);                      // spatial_attention_f32.cu: NMM_F32 flash kernel on the FMA pipe
int launch_spatial_attention_f32_tiled(const FlashArgs &a, cudaStream_t st);
int device_check();

// GEMM + epilogue
// Internal epilogue (not part of the C ABI enum): the QKV projection with the temporal attention fused into its epilogue --
// the tile's q | k | v never leave the SM (gemm_tcgen05.cu, "QKV + attention").
constexpr int NMM_EPI_QKV_ATTN = 4;
constexpr int NMM_ATTN_TILE_CH = 80;      // channels of q (and of k, v) per N tile of the fused kernel: 2 heads of 40 or 1 head of 80

struct LinearArgs {
    int epilogue;            // nmm_epilogue
    int64_t M;
    int N, K;                // N = rows of W
    const void *A;           // [M,K]  dtype
    const void *W;           // [N,K]  dtype
    const float *bias;       // [N] fp32 or null
    float *h;                // RESIDUAL: fp32 [M,N] in/out
    void *out;               // STORE: [M,N]; RESIDUAL: optional [M,N] copy; GEGLU: [M,N/2]   (dtype)
    int no_h_store;          // RESIDUAL: h is only read, the sum goes to `out` alone (the last feed-forward)
    int planes;              // 0 / 1: plain bf16.  2 (NMM_F32X3) / 3 (NMM_F32X6), tensor-core path only: A is bf16 [M, planes * K] and W bf16
                             // [N, planes * K], each row = hi | lo (| mid | lo) planes; `out` is written the same way ([M, planes * N], GEGLU
                             // [M, planes * N / 2]); x / y of the OUTPUT epilogue are fp32 (gemm_tcgen05.cu, PL)
    // OUTPUT epilogue
    const void *x; void *y;
    int F, P;
    int64_t xsb, xsc, xsf, ysb, ysc, ysf;
    float2 *y_part;          // OUTPUT epilogue (bf16 vector path), or null: [M / 32][N] (sum, sum of squares) of y as stored, per 32-row block and channel
    // GroupNorm-fused A operand (bf16 tensor-core path, STORE epilogue: proj_in).  A is NULL; the A tiles are TMA-loaded straight
    // from x [b, c, f, p] (channel rows of positions = an M-major operand), normalised in shared memory
    // (x * rstd*gamma[c] + beta[c] - mean*rstd*gamma[c], rounded to bf16 exactly like the stand-alone gn_tokens kernel) and fed to
    // the tensor core through an MN-major descriptor.  Uses F, P, xsb/xsc/xsf above; needs P % 64 == 0 and M % 128 == 0.
    const void *gn_x;
    const double *gn_partial; int gn_splits; double gn_count; float gn_eps;
    const float *gn_w, *gn_b;
    int gn_B;
    // NMM_EPI_QKV_ATTN: A = LayerNorm output tokens [M, K]; W = the q|k|v weight with rows regrouped per 80-channel tile
    // (q rows 80t..80t+79, then the k rows, then the v rows of the same channels); out = ctx [M, K].  Uses F, P above, attn_B
    // images and attn_heads; needs d_h in {40, 80}, F in {8, 16}, P % (128 / F) == 0.
    int attn_B, attn_heads;
    // LayerNorm folding (bf16 tensor-core path only; see gemm_tcgen05.cu "LayerNorm folding"):
    //   producer side: this GEMM writes the residual stream -> also emit per-row partial (sum, sum of squares) of the new h
    float *ln_part_out;      // [M][NMM_LN_PARTS][2] fp32 or null
    //   consumer side: A holds the RAW bf16 residual rows and W is gamma-folded; the epilogue applies
    //   out = rstd * (acc - mean * g[n]) + c[n] (+ pew[frame][n]) with mean / rstd from the partials of the producer
    const float *ln_part_in; // [M][NMM_LN_PARTS][2] or null
    int ln_nparts;           // valid partial slots per row (2 * n_tiles of the producer GEMM)
    const float *ln_g, *ln_c;   // [N] fp32: g[n] = sum_c W'[n,c];  c[n] = sum_c beta[c] W[n,c] + bias[n]
    const float *ln_pew;     // [max_len][N] fp32 or null: pe[f] . W^T
    float ln_eps;
};
constexpr int NMM_LN_PARTS = 16;     // partial-statistics slots per row: 2 epilogue warps x up to 8 N tiles of the producer
// N tile / CTA-pair plan the tensor-core GEMM will use for (M, N, K): lets the caller know how many partial-statistics slots
// a producer GEMM fills (2 * N / block_n)
int launch_gn_apply(const Geo &g, const nmm_shape *s, const void *x, void *y, const float *mean, const float *rstd, const float *gn_w,
                    const float *gn_b, int silu, cudaStream_t st);
int launch_cfg_ddim(int dtype, int64_t n, void *x, const void *eu, const void *ec, float g, double a_t, double a_prev, cudaStream_t st);
bool linear_tc_attn_fusable(int C, int heads, int F, int P);
bool linear_tc_gn_fusable(int64_t M, int P, const void *x, int64_t sb, int64_t sc, int64_t sf);
void plan_linear_tc(int64_t M, int N, int K, int epilogue, int *block_n, int *cluster);
// algorithmic work of one Linear launch (DESIGN.md section 4): 2*M*N*K flops; bytes = operands once + epilogue traffic once
inline double linear_flops(const LinearArgs &a) { return 2.0 * (double)a.M * a.N * a.K; }
inline double linear_bytes(const LinearArgs &a, int es) {
    const double MN = (double)a.M * a.N;
    double b = ((double)a.M * a.K + (double)a.N * a.K) * es + (a.bias ? 4.0 * a.N : 0.0);
    switch (a.epilogue) {
        case NMM_EPI_STORE: b += (a.h ? 4.0 * MN : 0.0) + (a.out ? es * MN : 0.0); break;
        case NMM_EPI_RESIDUAL: b += 4.0 * MN + (a.out ? es * MN : 4.0 * MN); break;
        case NMM_EPI_GEGLU: b += es * MN / 2; break;
        case NMM_EPI_QKV_ATTN: b += es * (double)a.M * a.K; break;      // only ctx is written

        default: b += 2.0 * es * MN; break;      // OUTPUT: read x, write y
    }
    return b;
}
// The whole module in one kernel (fused_module.cu): C = 320, 8 heads, 8 or 16 frames, bf16.
struct FusedArgs {
    const void *x; void *y;
    int64_t xsb, xsc, xsf, ysb, ysc, ysf;
    int B, F, P, A, pos_enc;
    const double *gn_partial; int gn_splits; double gn_count; float gn_eps;
    const void *w_in_g, *w_out, *w1, *w2;                   // packed bf16 weights (w_in_g: GroupNorm gamma folded in; w1 GEGLU-interleaved)
    const void *wqkv_t[NMM_MAX_ATTN], *wo[NMM_MAX_ATTN];    // q|k|v in head-pair tile order; to_out
    const void *wo_tail[NMM_MAX_ATTN];                      // to_out columns 64-79 of every head pair, un-swizzled operand layout
    const float *vec_attn[NMM_MAX_ATTN], *vec_ff, *vec_fin; // fp32 vector blocks (FmParams, fused_module.cu)
    const float *b1;
    float ln_eps;
    float *stage_dump; int stage_id;                         // tests: snapshot of the residual stream after stage stage_id (or null)
    float2 *y_part;                                          // or null: per (tile, frame, group) sums of y (N1: statistics for the next GroupNorm)
};
bool fused_module_weights(const Geo &g);
bool fused_module_eligible(const Geo &g, const nmm_shape *s, const void *x);
int launch_fused_module(const FusedArgs &a, cudaStream_t st);
int launch_linear_simt(const LinearArgs &a, cudaStream_t st);     // fp32
int launch_linear_tc(const LinearArgs &a, cudaStream_t st);       // bf16 tcgen05
int linear_dispatch(int dtype, const LinearArgs &a, cudaStream_t st);     // bf16 -> tcgen05, NMM_F32X3 / X6 -> tcgen05 3 / 6 x bf16, NMM_F32 -> FMA
// parameter packing
int launch_convert_rows(const void *src, int src_dtype, void *dst, int dst_dtype, int64_t rows, int64_t cols,
                        int interleave_half /*0 or rows/2*/, cudaStream_t st);

}  // namespace nmm

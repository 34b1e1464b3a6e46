// GroupNorm statistics, GroupNorm-apply fused with the (b f) c h w -> (b f)(h w) c re-layout, and
// LayerNorm(+positional encoding).  All three are HBM-bound streaming kernels (SURVEY 8(d)):
//   gn_stats        reads x once                                   bytes = N*C*s
//   gn_tokens       reads x once, writes tokens once               bytes = 2*N*C*s
//   layernorm_pe    reads h (fp32) once, writes n once             bytes = N*C*(4+s)
// Reference arithmetic: motion_module.py:142-144 (GroupNorm + permute/reshape), :212/:219 (LayerNorm),
// :241-243 (x + pe[:, :f]).
#include <type_traits>

#include "common.cuh"

namespace nmm {

// ------------------------------------------------------------------------------------------------
// GroupNorm statistics.  One (b,f,group) = cpg channels x P positions; each channel is a dense run of
// P elements at x + b*sb + c*sc + f*sf.  The group's cpg*P elements are cut into `splits` chunks so the
// grid has >= ~8 CTAs per SM; each CTA writes one (sum, sumsq) pair in double.  Finalisation (mean,
// rstd) is done by the consumer, so there are no atomics and the result is deterministic.
// ------------------------------------------------------------------------------------------------
// Launch shape: one CTA per (b, f, group, split); a CTA of TH threads keeps PT 16-byte loads per thread in flight (all issued before
// the first accumulate).  The plan picks the smallest (TH, PT) whose chunk TH * PT * 8 covers a whole group, so that at the UNet
// levels of the bench (10 x 4096, 20 x 1024, 40 x 256, 40 x 64 elements per group) a group is ONE CTA, the grid (B*F*32 CTAs) is a
// single wave with >= 64 KB of loads in flight per SM, and the consumers finalise from one partial per group.  (Round 1 used fixed
// 256 x 8 chunks: 1536 CTAs = 1.3 waves at the 64 x 64 level, 2.2 TB/s; the tail wave ran on a third of the machine.)
constexpr int GN_MAX_THREADS = 512, GN_MAX_PT = 16;
struct GnPlan { int threads, pt, splits; };
static GnPlan gn_plan(const Geo &g) {
    const int64_t total = (int64_t)(g.C / NMM_GN_GROUPS) * g.P;
    const int64_t cap = (int64_t)GN_MAX_THREADS * GN_MAX_PT * 8;
    GnPlan p;
    p.splits = (int)ceil_div(total, cap);
    const int64_t per = ceil_div(total, (int64_t)p.splits);            // elements one CTA must cover
    static const int TH[4] = {64, 128, 256, 512}, PT[5] = {4, 5, 8, 10, 16};
    int64_t best = -1;
    p.threads = GN_MAX_THREADS; p.pt = GN_MAX_PT;
    for (int t = 0; t < 4; t++)
        for (int q = 0; q < 5; q++) {
            const int64_t chunk = (int64_t)TH[t] * PT[q] * 8;
            if (chunk >= per && (best < 0 || chunk < best || (chunk == best && TH[t] > p.threads))) { best = chunk; p.threads = TH[t]; p.pt = PT[q]; }
        }
    return p;
}
static int gn_splits(const Geo &g) { return gn_plan(g).splits; }
int gn_splits_of(const Geo &g) { return gn_splits(g); }
size_t gn_partial_bytes(const Geo &g) {
    return (size_t)g.B * g.F * NMM_GN_GROUPS * gn_splits(g) * 2 * sizeof(double);
}

template <typename T> struct Vec16;   // 16-byte vector of T
template <> struct Vec16<float> { static constexpr int N = 4; };
template <> struct Vec16<bf16> { static constexpr int N = 8; };

// Accumulation of the 16 bytes of one vector on the packed fp32x2 pipe: d = v - K, s += d, ss += d * d with two accumulator lanes
// (even / odd elements of the vector), nK2 = (-K, -K) (K = 0 for bf16: d = v exactly).  Three packed instructions per element pair.
template <typename T>
__device__ __forceinline__ void accum16v(const uint4 v, uint64_t nK2, uint64_t &s2, uint64_t &ss2) {
    if constexpr (sizeof(T) == 4) {
        const uint64_t d0 = f32x2_add(f32x2_pack(__uint_as_float(v.x), __uint_as_float(v.y)), nK2);
        const uint64_t d1 = f32x2_add(f32x2_pack(__uint_as_float(v.z), __uint_as_float(v.w)), nK2);
        s2 = f32x2_add(s2, d0); ss2 = f32x2_fma(d0, d0, ss2);
        s2 = f32x2_add(s2, d1); ss2 = f32x2_fma(d1, d1, ss2);
    } else {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint64_t d = f32x2_add(f32x2_pack(bf16_lo(w[i]), bf16_hi(w[i])), nK2);
            s2 = f32x2_add(s2, d); ss2 = f32x2_fma(d, d, ss2);
        }
    }
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// VEC: PT 16-byte vectors per thread (chunk = blockDim.x * PT vectors); !VEC: element loop over the same chunk.
template <typename T, bool VEC, int PT>
__global__ void __launch_bounds__(GN_MAX_THREADS) gn_stats_kernel(const T *__restrict__ x, double *__restrict__ partial,
                                                                  int C, int F, int P, int splits, int64_t sb, int64_t sc,
                                                                  int64_t sf) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    const int cpg = C / NMM_GN_GROUPS;
    const int split = blockIdx.x % splits;
    const int grp = (blockIdx.x / splits) % NMM_GN_GROUPS;
    const int bf = blockIdx.x / (splits * NMM_GN_GROUPS);
    const int b = bf / F, f = bf % F;
    const T *base = x + (int64_t)b * sb + (int64_t)f * sf + (int64_t)grp * cpg * sc;
    const int64_t total = (int64_t)cpg * P;
    constexpr int V = Vec16<T>::N;
    const int64_t chunk = (int64_t)blockDim.x * PT * 8;                 // elements per CTA (8 = bf16 per vector; the fp32 path covers it in 2 PT rounds)
    const int64_t e0 = (int64_t)split * chunk;
    const int64_t e1 = min(total, e0 + chunk);
    // One-pass sums of x and x^2 lose (|mean| / std)^2 of relative accuracy in the variance once they are rounded, and the cancellation
    // in c2 / count - mean^2 comes after.  So each thread's fp32 sums go to double before any sum over threads, and:
    //  * fp32 input: every thread accumulates x - K, K = the fp32 mean of the first min(P, 8) elements of the group (the same value in
    //    every thread and split), which keeps the per-thread sums well conditioned whatever the offset;
    //  * bf16 input: no shift.  x^2 of a bf16 value has 16 significant bits, so a thread's fp32 sums of <= 128 of them are exact whenever
    //    the values share an exponent range -- which an offset group does -- and a shift would only add rounding.
    auto shift_of = [&]() {                            // broadcast loads (L1 / L2 after the first warp)
        if constexpr (sizeof(T) != 4) return 0.f;
        const int nk = P < 8 ? P : 8;
        float acc = 0.f;
        for (int j = 0; j < nk; j++) acc += to_f32(__ldg(base + j));
        return acc / (float)nk;
    };
    float K = 0.f;
    float s = 0.f, ss = 0.f;
    int n = 0;                                         // valid elements this thread accumulated
    if constexpr (VEC) {
        uint64_t s2 = f32x2_pack(0.f, 0.f), ss2 = s2, nK2 = s2;
        const int tot = (int)total;                    // cpg*P < 2^31 (validated); P % V == 0, so a vector never straddles channels
        constexpr int ROUNDS = 8 / V;                   // fp32: 4 elements per vector -> two rounds of PT loads cover the same chunk
#pragma unroll
        for (int rd = 0; rd < ROUNDS; rd++) {
            const int base_e = (int)e0 + rd * (int)blockDim.x * PT * V;
            // issue every load of this round before the first accumulate
            uint4 v[PT];
            uint32_t ok_mask = 0;
#pragma unroll
            for (int i = 0; i < PT; i++) {
                const int e = base_e + (i * (int)blockDim.x + (int)threadIdx.x) * V;
                const bool ok = e < tot;
                const int c = ok ? e / P : 0;
                const int p = ok ? e - c * P : 0;
                v[i] = ok ? __ldg(reinterpret_cast<const uint4 *>(base + (int64_t)c * sc + p)) : make_uint4(0u, 0u, 0u, 0u);
                ok_mask |= (uint32_t)ok << i;
            }
            if (rd == 0) {                              // once this round's loads are in flight
                K = shift_of();
                nK2 = f32x2_pack(-K, -K);
            }
#pragma unroll
            for (int i = 0; i < PT; i++)
                if (ok_mask >> i & 1u) { accum16v<T>(v[i], nK2, s2, ss2); n += V; }     // a lane past the group's end adds nothing, not (0 - K)^2
        }
        float a0, a1;
        f32x2_unpack(s2, a0, a1); s = a0 + a1;
        f32x2_unpack(ss2, a0, a1); ss = a0 + a1;
    } else {
        K = shift_of();
        for (int64_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            int c = (int)(e / P); int p = (int)(e - (int64_t)c * P);
            const float d = to_f32(base[(int64_t)c * sc + p]) - K;
            s += d; ss = fmaf(d, d, ss); n++;
        }
    }
    // un-shift per thread in double (s, ss, K are fp32 and n <= 128, so only double roundings remain), then reduce in double:
    //   sum x = s + n K,  sum x^2 = ss + 2 K s + n K^2
    __shared__ double sh[2][GN_MAX_THREADS / 32];
    const double dK = (double)K, dsh = (double)s;
    const double ds = warp_sum_d(fma((double)n, dK, dsh)), dss = warp_sum_d(fma((double)n * dK, dK, fma(2.0 * dK, dsh, (double)ss)));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { sh[0][warp] = ds; sh[1][warp] = dss; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, c2 = 0;
        const int nw = (int)blockDim.x >> 5;
        for (int i = 0; i < nw; i++) { a += sh[0][i]; c2 += sh[1][i]; }
        partial[(int64_t)blockIdx.x * 2 + 0] = a;
        partial[(int64_t)blockIdx.x * 2 + 1] = c2;
    }
}

template <typename T>
static bool x_vec_ok(const Geo &g, const nmm_shape *s, const void *x) {
    const int V = 16 / (int)sizeof(T);
    return g.P % V == 0 && s->x_stride_b % V == 0 && s->x_stride_c % V == 0 && s->x_stride_f % V == 0 && aligned(x, 16);
}

template <typename T, bool VEC>
static void launch_gn_stats_pt(const GnPlan &pl, dim3 grid, cudaStream_t st, const T *x, double *partial, const Geo &g, const nmm_shape *s) {
    const dim3 block((unsigned)pl.threads);
#define GN_PT(N) launch_pdl(gn_stats_kernel<T, VEC, N>, grid, block, 0, st, x, partial, g.C, g.F, g.P, pl.splits, s->x_stride_b, s->x_stride_c, s->x_stride_f)
    switch (pl.pt) {
        case 4: GN_PT(4); break;
        case 5: GN_PT(5); break;
        case 8: GN_PT(8); break;
        case 10: GN_PT(10); break;
        default: GN_PT(16); break;
    }
#undef GN_PT
}

int launch_gn_stats(const Geo &g, const nmm_shape *s, const void *x, double *partial, cudaStream_t st) {
    const GnPlan pl = gn_plan(g);
    const int64_t blocks = (int64_t)g.B * g.F * NMM_GN_GROUPS * pl.splits;
    if (blocks > 0x7fffffff) return fail(NMM_ERR_UNSUPPORTED, "gn_stats grid too large");
    dim3 grid((unsigned)blocks);
    ProfScope prof(K_GN_STATS, st, 0.0, (double)g.N * g.C * dtype_size(g.dtype));
    if (g.dtype == NMM_BF16) {
        if (x_vec_ok<bf16>(g, s, x)) launch_gn_stats_pt<bf16, true>(pl, grid, st, (const bf16 *)x, partial, g, s);
        else launch_gn_stats_pt<bf16, false>(pl, grid, st, (const bf16 *)x, partial, g, s);
    } else {
        if (x_vec_ok<float>(g, s, x)) launch_gn_stats_pt<float, true>(pl, grid, st, (const float *)x, partial, g, s);
        else launch_gn_stats_pt<float, false>(pl, grid, st, (const float *)x, partial, g, s);
    }
    NMM_LAUNCHED("gn_stats_kernel");
    return NMM_OK;
}

__global__ void gn_finalize_kernel(const double *__restrict__ partial, float *__restrict__ mean, float *__restrict__ rstd,
                                   int n, int splits, double count, float eps) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float m, r;
    gn_finalize_one(partial, i, splits, count, eps, m, r);
    mean[i] = m; rstd[i] = r;
}

int launch_gn_finalize(const Geo &g, const nmm_shape *s, const double *partial, float *mean, float *rstd, cudaStream_t st, int splits_override) {
    const int n = g.B * g.F * NMM_GN_GROUPS;
    launch_pdl(gn_finalize_kernel, (n + 127) / 128, 128, 0, st, partial, mean, rstd, n, splits_override > 0 ? splits_override : gn_splits(g),
                                                         (double)(g.C / NMM_GN_GROUPS) * g.P, s->eps_gn);
    NMM_LAUNCHED("gn_finalize_kernel");
    return NMM_OK;
}

// ------------------------------------------------------------------------------------------------
// GroupNorm apply + transpose to token-major.
//   tokens[(bf*P + p), c] = (x[b,c,f,p] - mean[bf,g]) * rstd[bf,g] * gamma[c] + beta[c]
// Generic kernel: 32(c) x 32(p) tile through shared memory, any dtype / alignment / ragged edges.
// ------------------------------------------------------------------------------------------------
// SPLIT = 2 (NMM_F32X3) / 3 (NMM_F32X6): tokens is a bf16 [N, SPLIT * C] tensor, every row = hi | lo (| mid | lo) planes of the fp32 values.
template <typename T, int SPLIT = 0>
__global__ void __launch_bounds__(256) gn_tokens_generic_kernel(const T *__restrict__ x, const double *__restrict__ partial,
                                                                const float *__restrict__ gamma, const float *__restrict__ beta,
                                                                T *__restrict__ tokens, int C, int F, int P, int splits, double count,
                                                                float eps, int64_t sb, int64_t sc, int64_t sf) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    __shared__ float tile[32][33];
    __shared__ float sc_a[32], sc_b[32];
    const int bf = blockIdx.z, b = bf / F, f = bf % F;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
    const int cpg = C / NMM_GN_GROUPS;
    if (threadIdx.x < 32) {
        int c = c0 + threadIdx.x;
        if (c < C) {
            float m, r;
            gn_finalize_one(partial, bf * NMM_GN_GROUPS + c / cpg, splits, count, eps, m, r);
            float a = r * gamma[c];
            sc_a[threadIdx.x] = a; sc_b[threadIdx.x] = beta[c] - m * a;
        }
    }
    __syncthreads();
    const T *base = x + (int64_t)b * sb + (int64_t)f * sf;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int cl = ty + i * 8, c = c0 + cl, p = p0 + tx;
        if (c < C && p < P) tile[cl][tx] = fmaf(to_f32(base[(int64_t)c * sc + p]), sc_a[cl], sc_b[cl]);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int pl = ty + i * 8, p = p0 + pl, c = c0 + tx;
        if (c < C && p < P) {
            if constexpr (SPLIT > 1) split1_store<SPLIT>(reinterpret_cast<bf16 *>(tokens) + ((int64_t)bf * P + p) * (SPLIT * C), C, c, tile[tx][pl]);
            else tokens[((int64_t)bf * P + p) * C + c] = from_f32<T>(tile[tx][pl]);
        }
    }
}

// Fast bf16 kernel: 64(c) x 64(p) tile, 16-byte loads along p, channel pairs packed as bf16x2 before the
// shared-memory transpose (4-byte conflict-light stores), 16-byte stores along c.  Requires C % 64 == 0,
// P % 64 == 0 and 16-byte aligned rows.
__global__ void __launch_bounds__(256) gn_tokens_bf16_kernel(const bf16 *__restrict__ x, const double *__restrict__ partial,
                                                             const float *__restrict__ gamma, const float *__restrict__ beta,
                                                             bf16 *__restrict__ tokens, int C, int F, int P, int splits, double count,
                                                             float eps, int64_t sb, int64_t sc, int64_t sf) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    __shared__ uint32_t tile[64][33];            // [p][channel pair]
    __shared__ float sc_a[64], sc_b[64];
    const int bf = blockIdx.z, b = bf / F, f = bf % F;
    const int c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
    const int cpg = C / NMM_GN_GROUPS;
    const int t = threadIdx.x;
    if (t < 64) {
        int c = c0 + t;
        float m, r;
        gn_finalize_one(partial, bf * NMM_GN_GROUPS + c / cpg, splits, count, eps, m, r);
        float a = r * gamma[c];
        sc_a[t] = a; sc_b[t] = beta[c] - m * a;
    }
    const int pv = t & 7, cp = t >> 3;           // 8 p-vectors x 32 channel pairs
    const bf16 *src = x + (int64_t)b * sb + (int64_t)f * sf + (int64_t)(c0 + 2 * cp) * sc + p0 + pv * 8;
    uint4 v0 = __ldg(reinterpret_cast<const uint4 *>(src));
    uint4 v1 = __ldg(reinterpret_cast<const uint4 *>(src + sc));
    __syncthreads();
    const float a0 = sc_a[2 * cp], b0 = sc_b[2 * cp], a1 = sc_a[2 * cp + 1], b1 = sc_b[2 * cp + 1];
    const uint32_t w0[4] = {v0.x, v0.y, v0.z, v0.w}, w1[4] = {v1.x, v1.y, v1.z, v1.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        tile[pv * 8 + 2 * i][cp] = pack_bf16x2(fmaf(bf16_lo(w0[i]), a0, b0), fmaf(bf16_lo(w1[i]), a1, b1));
        tile[pv * 8 + 2 * i + 1][cp] = pack_bf16x2(fmaf(bf16_hi(w0[i]), a0, b0), fmaf(bf16_hi(w1[i]), a1, b1));
    }
    __syncthreads();
    const int pl = t >> 2, q = t & 3;            // 64 rows x 4 quarter-rows (32 bytes each)
    uint32_t o[8];
#pragma unroll
    for (int i = 0; i < 8; i++) o[i] = tile[pl][q * 8 + i];
    bf16 *dst = tokens + ((int64_t)bf * P + p0 + pl) * C + c0 + q * 16;
    reinterpret_cast<uint4 *>(dst)[0] = make_uint4(o[0], o[1], o[2], o[3]);
    reinterpret_cast<uint4 *>(dst)[1] = make_uint4(o[4], o[5], o[6], o[7]);
}

// ------------------------------------------------------------------------------------------------
// SURVEY 8(f) N1: statistics of the module OUTPUT for the next InflatedGroupNorm (ResnetBlock3D.norm1, resnet.py:182-198;
// call order unet_blocks.py:407-411).  The last kernel of the module emits fp32 partial (sum, sum of squares) of y as stored;
// these kernels reduce them -- one warp per (b, f, group), fixed order, double accumulation, no atomics -- to the
// [B*F*32][2] double "sums" format every GroupNorm consumer of the library accepts as precomputed statistics.
// ------------------------------------------------------------------------------------------------
// part[tile][F][32] (fused module kernel; tile = b * tiles_per_b + tt)
__global__ void __launch_bounds__(256) y_sums_from_tiles_kernel(const float2 *__restrict__ part, double *__restrict__ sums, int F, int tiles_per_b, int n) {
    pdl_wait();
    pdl_launch_dependents();
    const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;                              // warp-uniform
    const int g = i % NMM_GN_GROUPS, bf = i / NMM_GN_GROUPS, b = bf / F, f = bf - b * F;
    double a = 0, c2 = 0;
    for (int tt = lane; tt < tiles_per_b; tt += 32) {
        const float2 v = __ldg(part + ((int64_t)(b * tiles_per_b + tt) * F + f) * NMM_GN_GROUPS + g);
        a += (double)v.x; c2 += (double)v.y;
    }
    a = warp_sum_d(a); c2 = warp_sum_d(c2);
    if (lane == 0) { sums[2 * (int64_t)i] = a; sums[2 * (int64_t)i + 1] = c2; }
}
// part[M / 32][C] (tensor-core GEMM, OUTPUT epilogue): image bf owns the row blocks [bf * P / 32, (bf + 1) * P / 32)
__global__ void __launch_bounds__(256) y_sums_from_channels_kernel(const float2 *__restrict__ part, double *__restrict__ sums, int C, int p32, int n) {
    pdl_wait();
    pdl_launch_dependents();
    const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const int cpg = C / NMM_GN_GROUPS, g = i % NMM_GN_GROUPS, bf = i / NMM_GN_GROUPS;
    double a = 0, c2 = 0;
    for (int it = lane; it < p32 * cpg; it += 32) {
        const int rb = it / cpg, c = g * cpg + (it - rb * cpg);
        const float2 v = __ldg(part + ((int64_t)bf * p32 + rb) * C + c);
        a += (double)v.x; c2 += (double)v.y;
    }
    a = warp_sum_d(a); c2 = warp_sum_d(c2);
    if (lane == 0) { sums[2 * (int64_t)i] = a; sums[2 * (int64_t)i + 1] = c2; }
}
// partial[n][splits][2] (gn_stats) -> sums[n][2]
__global__ void gn_partial_to_sums_kernel(const double *__restrict__ partial, double *__restrict__ sums, int n, int splits) {
    pdl_wait();
    pdl_launch_dependents();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double a = 0, c2 = 0;
    for (int k = 0; k < splits; k++) { a += partial[((int64_t)i * splits + k) * 2]; c2 += partial[((int64_t)i * splits + k) * 2 + 1]; }
    sums[2 * (int64_t)i] = a; sums[2 * (int64_t)i + 1] = c2;
}
int launch_y_sums_tiles(const float2 *part, double *sums, int B, int F, int tiles_per_b, cudaStream_t st) {
    const int n = B * F * NMM_GN_GROUPS;
    launch_pdl(y_sums_from_tiles_kernel, (unsigned)ceil_div((int64_t)n * 32, 256), 256, 0, st, part, sums, F, tiles_per_b, n);
    NMM_LAUNCHED("y_sums_from_tiles_kernel");
    return NMM_OK;
}
int launch_y_sums_channels(const float2 *part, double *sums, int BF, int C, int P, cudaStream_t st) {
    const int n = BF * NMM_GN_GROUPS;
    launch_pdl(y_sums_from_channels_kernel, (unsigned)ceil_div((int64_t)n * 32, 256), 256, 0, st, part, sums, C, P / 32, n);
    NMM_LAUNCHED("y_sums_from_channels_kernel");
    return NMM_OK;
}
int launch_gn_partial_to_sums(const Geo &g, const double *partial, double *sums, cudaStream_t st) {
    const int n = g.B * g.F * NMM_GN_GROUPS;
    launch_pdl(gn_partial_to_sums_kernel, (unsigned)ceil_div(n, 128), 128, 0, st, partial, sums, n, gn_splits(g));
    NMM_LAUNCHED("gn_partial_to_sums_kernel");
    return NMM_OK;
}

// `g` / `s` describe the positions being converted (possibly a chunk of the image: x already offset to its first position);
// `full` is the geometry the statistics were computed over (splits and element count of a whole group).
int launch_gn_tokens(const Geo &g, const nmm_shape *s, const Geo &full, const void *x, const double *partial, const float *gn_w,
                     const float *gn_b, void *tokens, cudaStream_t st, int splits_override) {
    const int splits = splits_override > 0 ? splits_override : gn_splits(full);
    const double count = (double)(full.C / NMM_GN_GROUPS) * full.P;
    if (g.B * g.F > 65535) return fail(NMM_ERR_UNSUPPORTED, "batch*frames > 65535");
    if (g.dtype == NMM_BF16 && g.C % 64 == 0 && g.P % 64 == 0 && x_vec_ok<bf16>(g, s, x) && aligned(tokens, 16)) {
        dim3 grid(g.P / 64, g.C / 64, g.B * g.F);
        ProfScope prof(K_GN_TOKENS, st, 0.0, 2.0 * g.N * g.C * dtype_size(g.dtype));
        launch_pdl(gn_tokens_bf16_kernel, grid, 256, 0, st, (const bf16 *)x, partial, gn_w, gn_b, (bf16 *)tokens, g.C, g.F, g.P,
                   splits, count, s->eps_gn, s->x_stride_b, s->x_stride_c, s->x_stride_f);
        NMM_LAUNCHED("gn_tokens_bf16_kernel");
        return NMM_OK;
    }
    dim3 grid((g.P + 31) / 32, (g.C + 31) / 32, g.B * g.F);
    if (grid.y > 65535) return fail(NMM_ERR_UNSUPPORTED, "channels too large");
    ProfScope prof(K_GN_TOKENS, st, 0.0, 2.0 * g.N * g.C * dtype_size(g.dtype));
    if (g.dtype == NMM_BF16)
        launch_pdl(gn_tokens_generic_kernel<bf16>, grid, 256, 0, st, (const bf16 *)x, partial, gn_w, gn_b, (bf16 *)tokens, g.C, g.F,
                   g.P, splits, count, s->eps_gn, s->x_stride_b, s->x_stride_c, s->x_stride_f);
    else if (g.dtype == NMM_F32X3)
        launch_pdl(gn_tokens_generic_kernel<float, 2>, grid, 256, 0, st, (const float *)x, partial, gn_w, gn_b, (float *)tokens, g.C, g.F,
                   g.P, splits, count, s->eps_gn, s->x_stride_b, s->x_stride_c, s->x_stride_f);
    else if (g.dtype == NMM_F32X6)
        launch_pdl(gn_tokens_generic_kernel<float, 3>, grid, 256, 0, st, (const float *)x, partial, gn_w, gn_b, (float *)tokens, g.C, g.F,
                   g.P, splits, count, s->eps_gn, s->x_stride_b, s->x_stride_c, s->x_stride_f);
    else
        launch_pdl(gn_tokens_generic_kernel<float>, grid, 256, 0, st, (const float *)x, partial, gn_w, gn_b, (float *)tokens, g.C, g.F,
                   g.P, splits, count, s->eps_gn, s->x_stride_b, s->x_stride_c, s->x_stride_f);
    NMM_LAUNCHED("gn_tokens_generic_kernel");
    return NMM_OK;
}

// ------------------------------------------------------------------------------------------------
// InflatedGroupNorm (+ optional SiLU) in place of layout: y[b,c,f,p] = act(GroupNorm per (b,f) image of x) -- the norm1 / norm2 +
// nonlinearity of ResnetBlock3D either side of the motion module (animatediff/models/resnet.py:21-29,182-198; SURVEY 8(f) N1).
// The reference rearranges b c f h w -> (b f) c h w (a copy), normalises, and rearranges back (another copy); here x is read in
// its own strides and y written in its own strides: 2 passes over x (statistics, apply) instead of ~6.
// ------------------------------------------------------------------------------------------------
constexpr int GNA_CHUNK = 4096;       // elements of one (b, f) image per CTA

__device__ __forceinline__ float silu_f(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

template <typename T, bool VEC, bool SILU>
__global__ void __launch_bounds__(256) gn_apply_kernel(const T *__restrict__ x, T *__restrict__ y, const float *__restrict__ mean,
                                                       const float *__restrict__ rstd, const float *__restrict__ gamma,
                                                       const float *__restrict__ beta, int C, int F, int P, int64_t xsb, int64_t xsc, int64_t xsf,
                                                       int64_t ysb, int64_t ysc, int64_t ysf) {
    pdl_wait();
    pdl_launch_dependents();
    const int bf = blockIdx.y, b = bf / F, f = bf - b * F;
    const int cpg = C / NMM_GN_GROUPS;
    const int64_t total = (int64_t)C * P;
    const T *xb = x + (int64_t)b * xsb + (int64_t)f * xsf;
    T *yb = y + (int64_t)b * ysb + (int64_t)f * ysf;
    constexpr int V = VEC ? 16 / (int)sizeof(T) : 1;
    for (int64_t e = ((int64_t)blockIdx.x * GNA_CHUNK) + (int64_t)threadIdx.x * V; e < min(total, ((int64_t)blockIdx.x + 1) * GNA_CHUNK); e += 256 * V) {
        const int c = (int)(e / P), p = (int)(e - (int64_t)c * P);
        const int gi = bf * NMM_GN_GROUPS + c / cpg;
        const float a = __ldg(rstd + gi) * __ldg(gamma + c);
        const float bb = __ldg(beta + c) - __ldg(mean + gi) * a;
        if constexpr (VEC) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(xb + (int64_t)c * xsc + p));
            uint4 o;
            if constexpr (sizeof(T) == 4) {
                float r[4] = {__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w)};
#pragma unroll
                for (int i = 0; i < 4; i++) { r[i] = fmaf(r[i], a, bb); if (SILU) r[i] = silu_f(r[i]); }
                o = make_uint4(__float_as_uint(r[0]), __float_as_uint(r[1]), __float_as_uint(r[2]), __float_as_uint(r[3]));
            } else {
                const uint32_t w[4] = {v.x, v.y, v.z, v.w};
                uint32_t ow[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    float lo = fmaf(bf16_lo(w[i]), a, bb), hi = fmaf(bf16_hi(w[i]), a, bb);
                    if (SILU) { lo = silu_f(lo); hi = silu_f(hi); }
                    ow[i] = pack_bf16x2(lo, hi);
                }
                o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            }
            *reinterpret_cast<uint4 *>(yb + (int64_t)c * ysc + p) = o;
        } else {
            float r = fmaf(to_f32(xb[(int64_t)c * xsc + p]), a, bb);
            if (SILU) r = silu_f(r);
            yb[(int64_t)c * ysc + p] = from_f32<T>(r);
        }
    }
}

int launch_gn_apply(const Geo &g, const nmm_shape *s, const void *x, void *y, const float *mean, const float *rstd, const float *gn_w,
                    const float *gn_b, int silu, cudaStream_t st) {
    if (g.B * g.F > 65535) return fail(NMM_ERR_UNSUPPORTED, "batch*frames > 65535");
    const int64_t chunks = ceil_div((int64_t)g.C * g.P, GNA_CHUNK);
    if (chunks > 0x7fffffff) return fail(NMM_ERR_UNSUPPORTED, "gn_apply grid too large");
    const dim3 grid((unsigned)chunks, (unsigned)(g.B * g.F));
    const int es = (int)dtype_size(g.dtype), V = 16 / es;
    const bool vec = g.P % V == 0 && GNA_CHUNK % (256 * V) == 0 && aligned(x, 16) && aligned(y, 16) && s->x_stride_b % V == 0 && s->x_stride_c % V == 0 &&
                     s->x_stride_f % V == 0 && s->y_stride_b % V == 0 && s->y_stride_c % V == 0 && s->y_stride_f % V == 0;
    ProfScope prof(K_GN_TOKENS, st, 0.0, 2.0 * g.N * g.C * es);
#define GNA_CASE(T, VV, SS)                                                                                                          \
    launch_pdl(gn_apply_kernel<T, VV, SS>, grid, 256, 0, st, (const T *)x, (T *)y, mean, rstd, gn_w, gn_b, g.C, g.F, g.P, s->x_stride_b,  \
               s->x_stride_c, s->x_stride_f, s->y_stride_b, s->y_stride_c, s->y_stride_f)
    if (g.dtype == NMM_BF16) {
        if (vec) { if (silu) GNA_CASE(bf16, true, true); else GNA_CASE(bf16, true, false); }
        else { if (silu) GNA_CASE(bf16, false, true); else GNA_CASE(bf16, false, false); }
    } else {
        if (vec) { if (silu) GNA_CASE(float, true, true); else GNA_CASE(float, true, false); }
        else { if (silu) GNA_CASE(float, false, true); else GNA_CASE(float, false, false); }
    }
#undef GNA_CASE
    NMM_LAUNCHED("gn_apply_kernel");
    return NMM_OK;
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over C (+ pe[frame of the token]).  h is the fp32 residual stream; out is the GEMM operand dtype.
// Vector kernel: one 16-lane half-warp per token row, the row lives in registers as IT4 = C/64 float4 per lane
// (two-pass mean / variance in fp32), every global access is 16 bytes per lane.  Generic kernel: one warp per row, any C.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float half_warp_sum(float v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct SplitOut { uint32_t pair; };      // tag (4 bytes per element like fp32): `out` is bf16 [N, 2C], row = hi plane | lo plane (NMM_F32X3)
struct Split3Out { uint16_t t[3]; };     // tag (6 bytes per element): `out` is bf16 [N, 3C], row = hi | mid | lo planes (NMM_F32X6)
template <typename TOut> constexpr int split_planes_of() { return std::is_same<TOut, SplitOut>::value ? 2 : std::is_same<TOut, Split3Out>::value ? 3 : 0; }

template <typename TOut, int IT4>
__global__ void __launch_bounds__(256) layernorm_pe_vec_kernel(const float *__restrict__ h, const float *__restrict__ gamma,
                                                               const float *__restrict__ beta, const float *__restrict__ pe,
                                                               TOut *__restrict__ out, int64_t N, int F, int P, float eps) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    constexpr int C = IT4 * 64;
    const int l16 = threadIdx.x & 15;
    int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 4) + (threadIdx.x >> 4);
    const bool valid = row < N;
    if (!valid) row = N - 1;                         // keep the whole warp in the shuffles; stores are predicated
    const float4 *hr = reinterpret_cast<const float4 *>(h + row * C);
    float4 v[IT4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < IT4; i++) {
        v[i] = __ldg(hr + l16 + 16 * i);
        s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
    const float mu = half_warp_sum(s) * (1.0f / C);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < IT4; i++) {
        const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
        ss = fmaf(a, a, ss); ss = fmaf(b, b, ss); ss = fmaf(c, c, ss); ss = fmaf(d, d, ss);
    }
    const float rstd = rsqrtf(half_warp_sum(ss) * (1.0f / C) + eps);
    const float4 *per = pe ? reinterpret_cast<const float4 *>(pe + (int64_t)((row / P) % F) * C) : nullptr;
    TOut *orow = out + row * C;               // (SplitOut / Split3Out: 4 / 6 bytes per element, so this is the row's hi plane)
#pragma unroll
    for (int i = 0; i < IT4; i++) {
        const int c4 = l16 + 16 * i;
        const float4 gm = __ldg(reinterpret_cast<const float4 *>(gamma) + c4);
        const float4 bt = __ldg(reinterpret_cast<const float4 *>(beta) + c4);
        float4 o;
        o.x = fmaf((v[i].x - mu) * rstd, gm.x, bt.x); o.y = fmaf((v[i].y - mu) * rstd, gm.y, bt.y);
        o.z = fmaf((v[i].z - mu) * rstd, gm.z, bt.z); o.w = fmaf((v[i].w - mu) * rstd, gm.w, bt.w);
        if (per) { const float4 pp = __ldg(per + c4); o.x += pp.x; o.y += pp.y; o.z += pp.z; o.w += pp.w; }
        if (valid) {
            if constexpr (split_planes_of<TOut>() > 1) split4_store<split_planes_of<TOut>()>(reinterpret_cast<bf16 *>(orow), C, 4 * c4, o.x, o.y, o.z, o.w);
            else if constexpr (sizeof(TOut) == 2) reinterpret_cast<uint2 *>(orow)[c4] = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
            else reinterpret_cast<float4 *>(orow)[c4] = o;
        }
    }
}

template <typename TOut>
__global__ void __launch_bounds__(256) layernorm_pe_generic_kernel(const float *__restrict__ h, const float *__restrict__ gamma,
                                                                   const float *__restrict__ beta, const float *__restrict__ pe,
                                                                   TOut *__restrict__ out, int64_t N, int C, int F, int P, float eps) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= N) return;                            // warp-uniform
    const float *hr = h + row * C;
    const float *per = pe ? pe + (int64_t)((row / P) % F) * C : nullptr;
    TOut *orow = out + row * C;
    const float invC = 1.0f / (float)C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += hr[c];
    const float mu = warp_sum(s) * invC;
    float ss = 0.f;
    for (int c = lane; c < C; c += 32) { float a = hr[c] - mu; ss = fmaf(a, a, ss); }
    const float rstd = rsqrtf(warp_sum(ss) * invC + eps);
    for (int c = lane; c < C; c += 32) {
        float a = fmaf((hr[c] - mu) * rstd, gamma[c], beta[c]);
        if (per) a += per[c];
        if constexpr (split_planes_of<TOut>() > 1) split1_store<split_planes_of<TOut>()>(reinterpret_cast<bf16 *>(orow), C, c, a);
        else orow[c] = from_f32<TOut>(a);
    }
}

template <typename TOut>
static int launch_ln_t(const Geo &g, const nmm_shape *s, const float *h, const float *w, const float *b, const float *pe,
                       TOut *out, cudaStream_t st) {
    ProfScope prof(K_LAYERNORM, st, 0.0, (double)g.N * g.C * (4 + sizeof(TOut)));
    const bool vec_ok = aligned(h, 16) && aligned(w, 16) && aligned(b, 16) && aligned(out, 16) && (pe == nullptr || aligned(pe, 16));
    if (vec_ok && (g.C == 320 || g.C == 640 || g.C == 1280)) {
        // 16 rows (half-warps) per 256-thread CTA; at the small UNet levels fewer rows per CTA so that the grid still covers the
        // 148 SMs several times over (1024 tokens in 16-row CTAs would be 64 CTAs)
        int threads = 256;
        while (threads > 64 && ceil_div(g.N, threads / 16) < 4 * 148) threads >>= 1;
        const int64_t blocks = ceil_div(g.N, threads / 16);
        if (blocks > 0x7fffffff) return fail(NMM_ERR_UNSUPPORTED, "too many tokens");
        dim3 grid((unsigned)blocks), block((unsigned)threads);
        if (g.C == 320) launch_pdl(layernorm_pe_vec_kernel<TOut, 5>, grid, block, 0, st, h, w, b, pe, out, g.N, g.F, g.P, s->eps_ln);
        else if (g.C == 640) launch_pdl(layernorm_pe_vec_kernel<TOut, 10>, grid, block, 0, st, h, w, b, pe, out, g.N, g.F, g.P, s->eps_ln);
        else launch_pdl(layernorm_pe_vec_kernel<TOut, 20>, grid, block, 0, st, h, w, b, pe, out, g.N, g.F, g.P, s->eps_ln);
    } else {
        const int64_t blocks = ceil_div(g.N, 8);
        if (blocks > 0x7fffffff) return fail(NMM_ERR_UNSUPPORTED, "too many tokens");
        launch_pdl(layernorm_pe_generic_kernel<TOut>, (unsigned)blocks, 256, 0, st, h, w, b, pe, out, g.N, g.C, g.F, g.P, s->eps_ln);
    }
    NMM_LAUNCHED("layernorm_pe_kernel");
    return NMM_OK;
}

int launch_layernorm_pe(const Geo &g, const nmm_shape *s, const float *h, const float *w, const float *b, const float *pe,
                        void *out, cudaStream_t st) {
    if (g.dtype == NMM_BF16) return launch_ln_t<bf16>(g, s, h, w, b, pe, (bf16 *)out, st);
    if (g.dtype == NMM_F32X3) return launch_ln_t<SplitOut>(g, s, h, w, b, pe, (SplitOut *)out, st);
    if (g.dtype == NMM_F32X6) return launch_ln_t<Split3Out>(g, s, h, w, b, pe, (Split3Out *)out, st);
    return launch_ln_t<float>(g, s, h, w, b, pe, (float *)out, st);
}

}  // namespace nmm

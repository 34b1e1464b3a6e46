// fp32 spatial attention on the FMA pipe, flash-style (NMM_F32 above the crossover of launch_spatial_attention, spatial_attention.cu):
//     O = softmax(Q K^T * d_h^-1/2) V      per (image, head), fp32 throughout, no bf16 rounding anywhere
// The arithmetic is the checker's (spatial_attention_f32_kernel): the scale is folded into q, a score is one fmaf chain over d = 0 .. d_h - 1
// (so the scores are bit-identical to the checker's), weights are expf(s - running max), O and l are rescaled online by expf(m_old - m_new)
// and O is divided by l at the end.  What differs is the order in which the keys are summed.
//
// One CTA = BM queries of one (image, head), 128 threads as RG row groups x CG column groups (CG = d_h / 5: 8 / 16 / 32, lanes of one
// warp).  A thread owns R = 8 query rows (rg + RG * i) in both phases, so its rows' running max, rescale factor and row sum stay in
// registers:
//   S = Q K^T   the thread's 8 rows x KPT keys (cg + CG * kk) of a 32-key tile, float4 reads of Q and K rows along d
//   softmax     row max over the CG threads of a row by shuffles; weights to shared memory (P, row-major); partial row sums per thread
//   O += P V    the thread's 8 rows x 5 columns (cg + CG * j) of O in registers, float4 reads of P along the keys
// Q, K and V are row-major in shared memory (pitch d_h + 4 floats: the rows a warp reads together fall on distinct bank quads), K / V tiles
// stream through a double-buffered cp.async ring.  q, k, v are column slices of projection outputs (free row / image strides), the kv
// image of q image i is i / kv_div (the 77-token text cross-attention); ragged last tiles are zero-filled and masked.
#include "common.cuh"

namespace nmm {
namespace {

__device__ __forceinline__ void f32_cp_async16(uint32_t saddr, const void *g, bool valid) {
    const int sz = valid ? 16 : 0;      // src-size 0: the 16 bytes are zero-filled, nothing is read
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(sz) : "memory");
}
__device__ __forceinline__ void f32_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void f32_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int DH>
struct F32TileCfg {
    static constexpr int THREADS = 128;
    static constexpr int CG = DH / 5;               // threads sharing a query row: 8 / 16 / 32
    static constexpr int RG = THREADS / CG;
    static constexpr int R = 8;                     // query rows per thread
    static constexpr int BM = R * RG;               // queries per CTA: 128 / 64 / 32
    static constexpr int BN = 32;                   // keys per tile
    static constexpr int KPT = BN / CG;             // keys per thread in S = Q K^T: 4 / 2 / 1
    static constexpr int NC = DH / CG;              // columns of O per thread: 5
    static constexpr int PITCH = DH + 4;            // floats per Q / K / V row in shared memory
    static constexpr int PP = BN + CG;              // floats per P row: the rows a warp writes together start 8 / 16 / 32 banks apart
    static constexpr int CH = DH / 4;               // 16-byte chunks per row
    static constexpr int Q_FLOATS = BM * PITCH, KV_FLOATS = BN * PITCH, P_FLOATS = BM * PP;
    static constexpr int SMEM = 4 * (Q_FLOATS + 4 * KV_FLOATS + P_FLOATS);     // Q | K stage 0, 1 | V stage 0, 1 | P
    static constexpr int MIN_BLOCKS = DH == 160 ? 2 : 3;                        // 64 / 75 / 110.5 KB of shared memory per CTA
    static_assert(CG * NC == DH && CG * KPT == BN && 32 % CG == 0 && THREADS % CG == 0, "F32TileCfg");
};

}  // namespace

template <int DH>
__global__ void __launch_bounds__(128, F32TileCfg<DH>::MIN_BLOCKS) spatial_attention_f32_tiled_kernel(const FlashArgs a) {
    using Cfg = F32TileCfg<DH>;
    constexpr int THREADS = Cfg::THREADS, CG = Cfg::CG, RG = Cfg::RG, R = Cfg::R, BM = Cfg::BM, BN = Cfg::BN, KPT = Cfg::KPT, NC = Cfg::NC;
    constexpr int PITCH = Cfg::PITCH, PP = Cfg::PP, CH = Cfg::CH;
    extern __shared__ __align__(16) float f32_smem[];
    float *const sQ = f32_smem, *const sK = sQ + Cfg::Q_FLOATS, *const sV = sK + 2 * Cfg::KV_FLOATS, *const sP = sV + 2 * Cfg::KV_FLOATS;
    pdl_wait();
    pdl_launch_dependents();
    const int tid = threadIdx.x, cg = tid % CG, rg = tid / CG;
    const int q0 = blockIdx.x * BM, head = blockIdx.y, img = blockIdx.z;
    const int kv_img = img / a.kv_div;
    const float *qg = (const float *)a.q + (int64_t)img * a.q_bs + head * DH;
    const float *kg = (const float *)a.k + (int64_t)kv_img * a.kv_bs + head * DH;
    const float *vg = (const float *)a.v + (int64_t)kv_img * a.kv_bs + head * DH;
    const int Lq = a.Lq, Lkv = a.Lkv;
    const uint32_t sq = (uint32_t)__cvta_generic_to_shared(sQ), sk0 = (uint32_t)__cvta_generic_to_shared(sK),
                   sv0 = (uint32_t)__cvta_generic_to_shared(sV);

    for (int i = tid; i < BM * CH; i += THREADS) {
        const int r = i / CH, c = i - r * CH, row = q0 + r;
        const bool ok = row < Lq;
        f32_cp_async16(sq + (uint32_t)(r * PITCH + c * 4) * 4, qg + (int64_t)(ok ? row : 0) * a.q_rs + c * 4, ok);
    }
    f32_cp_async_commit();
    auto load_kv = [&](int t, int stage) {
        const uint32_t so = (uint32_t)(stage * Cfg::KV_FLOATS) * 4;
        for (int i = tid; i < BN * CH; i += THREADS) {
            const int r = i / CH, c = i - r * CH, key = t * BN + r;
            const bool ok = key < Lkv;
            const int64_t off = (int64_t)(ok ? key : 0) * a.kv_rs + c * 4;
            const uint32_t s = so + (uint32_t)(r * PITCH + c * 4) * 4;
            f32_cp_async16(sk0 + s, kg + off, ok);
            f32_cp_async16(sv0 + s, vg + off, ok);
        }
    };
    const int nt = (Lkv + BN - 1) / BN;
    load_kv(0, 0);
    f32_cp_async_commit();
    f32_cp_async_wait<1>();
    __syncthreads();
    // the checker's convention: q * scale first, then the dot product (the loop's first barrier publishes the scaled rows)
    for (int i = tid; i < BM * DH; i += THREADS) {
        const int r = i / DH;
        sQ[r * PITCH + (i - r * DH)] *= a.scale;
    }

    float o[R][NC], m[R], l[R];
#pragma unroll
    for (int i = 0; i < R; i++) {
        m[i] = -INFINITY; l[i] = 0.f;
#pragma unroll
        for (int j = 0; j < NC; j++) o[i][j] = 0.f;
    }
    for (int t = 0; t < nt; t++) {
        f32_cp_async_wait<0>();
        __syncthreads();                  // tile t landed for everyone; everyone is done with tile t - 1 (the other stage) and with P
        if (t + 1 < nt) load_kv(t + 1, (t + 1) & 1);
        f32_cp_async_commit();
        const float *K = sK + (t & 1) * Cfg::KV_FLOATS, *V = sV + (t & 1) * Cfg::KV_FLOATS;

        // ---- S = Q K^T: one fmaf chain per score over d = 0 .. d_h - 1 ----
        float s[R][KPT];
#pragma unroll
        for (int i = 0; i < R; i++)
#pragma unroll
            for (int kk = 0; kk < KPT; kk++) s[i][kk] = 0.f;
#pragma unroll
        for (int d = 0; d < DH; d += 4) {
            float4 kf[KPT];
#pragma unroll
            for (int kk = 0; kk < KPT; kk++) kf[kk] = *reinterpret_cast<const float4 *>(K + (cg + CG * kk) * PITCH + d);
#pragma unroll
            for (int i = 0; i < R; i++) {
                const float4 qf = *reinterpret_cast<const float4 *>(sQ + (rg + RG * i) * PITCH + d);
#pragma unroll
                for (int kk = 0; kk < KPT; kk++) {
                    float acc = s[i][kk];
                    acc = fmaf(qf.x, kf[kk].x, acc); acc = fmaf(qf.y, kf[kk].y, acc);
                    acc = fmaf(qf.z, kf[kk].z, acc); acc = fmaf(qf.w, kf[kk].w, acc);
                    s[i][kk] = acc;
                }
            }
        }
        const int key0 = t * BN;
        if (key0 + BN > Lkv) {            // keys past the end of a ragged last tile
#pragma unroll
            for (int kk = 0; kk < KPT; kk++)
                if (key0 + cg + CG * kk >= Lkv)
#pragma unroll
                    for (int i = 0; i < R; i++) s[i][kk] = -INFINITY;
        }
        // ---- online softmax: the tile's key 0 is valid, so every row's new max is finite ----
#pragma unroll
        for (int i = 0; i < R; i++) {
            float mx = m[i];
#pragma unroll
            for (int kk = 0; kk < KPT; kk++) mx = fmaxf(mx, s[i][kk]);
#pragma unroll
            for (int off = 1; off < CG; off <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            const float al = expf(m[i] - mx);
            m[i] = mx;
            float sum = 0.f;
            float *prow = sP + (rg + RG * i) * PP + cg;
#pragma unroll
            for (int kk = 0; kk < KPT; kk++) {
                const float e = expf(s[i][kk] - mx);
                prow[CG * kk] = e;
                sum += e;
            }
            l[i] = l[i] * al + sum;       // this thread's keys only; the CG partial sums of a row are added once at the end
#pragma unroll
            for (int j = 0; j < NC; j++) o[i][j] *= al;
        }
        __syncthreads();                  // P complete
        // ---- O += P V ----
#pragma unroll 2
        for (int k4 = 0; k4 < BN; k4 += 4) {
            float4 p[R];
#pragma unroll
            for (int i = 0; i < R; i++) p[i] = *reinterpret_cast<const float4 *>(sP + (rg + RG * i) * PP + k4);
#pragma unroll
            for (int kk = 0; kk < 4; kk++) {
                float vv[NC];
#pragma unroll
                for (int j = 0; j < NC; j++) vv[j] = V[(k4 + kk) * PITCH + cg + CG * j];
#pragma unroll
                for (int i = 0; i < R; i++) {
                    const float pk = kk == 0 ? p[i].x : kk == 1 ? p[i].y : kk == 2 ? p[i].z : p[i].w;
#pragma unroll
                    for (int j = 0; j < NC; j++) o[i][j] = fmaf(pk, vv[j], o[i][j]);
                }
            }
        }
    }
    float *og = (float *)a.o + (int64_t)img * a.o_bs + head * DH;
#pragma unroll
    for (int i = 0; i < R; i++) {
        float li = l[i];
#pragma unroll
        for (int off = 1; off < CG; off <<= 1) li += __shfl_xor_sync(0xffffffffu, li, off);
        const int row = q0 + rg + RG * i;
        if (row < Lq) {
#pragma unroll
            for (int j = 0; j < NC; j++) og[(int64_t)row * a.o_rs + cg + CG * j] = o[i][j] / li;
        }
    }
}

bool spatial_attention_f32_tiled_eligible(const FlashArgs &a) {
    // 16-byte cp.async rows: aligned slices, strides in whole float4s
    return a.dtype == NMM_F32 && (a.dh == 40 || a.dh == 80 || a.dh == 160) && aligned(a.q, 16) && aligned(a.k, 16) && aligned(a.v, 16) &&
           a.q_rs % 4 == 0 && a.kv_rs % 4 == 0 && a.q_bs % 4 == 0 && a.kv_bs % 4 == 0;
}

template <int DH>
static int launch_f32_tiled(const FlashArgs &a, cudaStream_t st) {
    using Cfg = F32TileCfg<DH>;
    static DeviceOnce once;
    NMM_CUDA_OK(once.max_smem(spatial_attention_f32_tiled_kernel<DH>, Cfg::SMEM));
    const dim3 grid((unsigned)ceil_div(a.Lq, Cfg::BM), (unsigned)a.heads, (unsigned)a.images);
    const double per = (double)a.images * a.heads;
    ProfScope prof(K_SPATIAL_ATTN, st, 4.0 * per * a.Lq * (double)a.Lkv * DH, 4.0 * (2.0 * per * a.Lq * DH + 2.0 * per / a.kv_div * a.Lkv * DH));
    NMM_CUDA_OK(launch_pdl(spatial_attention_f32_tiled_kernel<DH>, grid, dim3(Cfg::THREADS), (size_t)Cfg::SMEM, st, a));
    NMM_LAUNCHED("spatial_attention_f32_tiled_kernel");
    return NMM_OK;
}

int launch_spatial_attention_f32_tiled(const FlashArgs &a, cudaStream_t st) {
    switch (a.dh) {
        case 40: return launch_f32_tiled<40>(a, st);
        case 80: return launch_f32_tiled<80>(a, st);
        case 160: return launch_f32_tiled<160>(a, st);
        default: return fail(NMM_ERR_UNSUPPORTED, "fp32 tiled spatial attention: head dim %d not supported (40, 80, 160)", a.dh);
    }
}

}  // namespace nmm

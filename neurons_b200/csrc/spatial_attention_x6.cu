// fp32-EXACT spatial attention on the tensor cores (SURVEY 8(f) N3, NMM_F32X6 mode of the spatial transformer): the kernel of
// spatial_attention_x3.cu with every operand as a three-term bf16 split, x = hi + mid + lo + O(2^-24 |x|), and six MMAs per product
//     S  = Ql Kh + Qm Km + Qh Kl + Qm Kh + Qh Km + Qh Kh        O += Pl Vh + Pm Vm + Ph Vl + Pm Vh + Ph Vm + Ph Vh
// (every cross product of weight >= 2^-16, small terms first; mid.lo, lo.mid and lo.lo are <= 2^-24 and dropped; S and each 32-key tile's
// P V from zero in the MMA, the running O in round-to-nearest fp32 fmas), like
// the 6 x bf16 Linear layers (gemm_tcgen05.cu, PL = 3).  q, k, v arrive as bf16 planes -- row = hi | mid | lo, the format
// launch_convert_rows(..., NMM_F32X6) writes; the softmax weights are split in registers, the row sums add the fp32 weights, O leaves as fp32.
// Exponents as in the FMA-pipe kernels (spatial_attention_f32.cu): the running max m is kept in unscaled score units and a weight is
// expf((s - m) * scale), so the argument's rounding error is relative to s - m rather than to s, and the accuracy does not fall with the
// logit scale (x3 splits keep ~16 bits; its error grows with max |logit|).
// One CTA = 64 queries of one (image, head), 4 warps of 16 rows; 32-key stages (hi, mid, lo tiles of K and V: 6 tiles per stage,
// double-buffered cp.async) -- half the x3 kernel's key tile, so that the three Q planes plus two stages stay at 46 / 99 / 189 KB of shared
// memory for d_h 40 / 80 / 160 (4 / 2 / 1 CTAs per SM).  Reference arithmetic: CrossAttention._attention, motion_module_new.py:258-287 in fp32.
#include "attention_core.cuh"
#include "common.cuh"

namespace nmm {

constexpr int F6_BM = 64, F6_BN = 32, F6_THREADS = 128;

template <int DH>
struct F6Cfg {
    static constexpr int PITCH = ((DH / 8) % 2 == 1) ? DH : DH + 8;     // bf16 elements per shared-memory row (ldmatrix conflict-free)
    static constexpr int CH = DH / 8;
    static constexpr int QTILE = F6_BM * PITCH * 2;                     // one 64-row bf16 Q plane
    static constexpr int KTILE = F6_BN * PITCH * 2;                     // one 32-row bf16 K or V plane
    static constexpr int SMEM = 3 * QTILE + 2 * 6 * KTILE;              // Qh Qm Ql | stage 0: Kh Km Kl Vh Vm Vl | stage 1: ...
    static constexpr int KS16 = DH / 16;
    static constexpr bool TAIL8 = (DH % 16) == 8;
    static constexpr int NT = DH / 8;
    static constexpr bool QRES = DH <= 80;                              // Q fragments (three planes) resident in registers; d_h = 160 reloads them
};

__device__ __forceinline__ void f6_cp16(uint32_t saddr, const void *g, bool valid) {
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(sz) : "memory");
}

// d += the six products of (a plane p, b plane p') in the order of the file header; a[p] / b[p]: fragments of plane p (0 hi, 1 mid, 2 lo)
__device__ __forceinline__ void mma6_k16(float (&d)[4], const uint32_t (&a)[3][4], const uint32_t (&b)[3][2]) {
    mma_k16(d, a[2][0], a[2][1], a[2][2], a[2][3], b[0][0], b[0][1]);
    mma_k16(d, a[1][0], a[1][1], a[1][2], a[1][3], b[1][0], b[1][1]);
    mma_k16(d, a[0][0], a[0][1], a[0][2], a[0][3], b[2][0], b[2][1]);
    mma_k16(d, a[1][0], a[1][1], a[1][2], a[1][3], b[0][0], b[0][1]);
    mma_k16(d, a[0][0], a[0][1], a[0][2], a[0][3], b[1][0], b[1][1]);
    mma_k16(d, a[0][0], a[0][1], a[0][2], a[0][3], b[0][0], b[0][1]);
}
__device__ __forceinline__ void mma6_k8(float (&d)[4], const uint32_t (&a)[3][2], const uint32_t (&b)[3]) {
    mma_k8(d, a[2][0], a[2][1], b[0]);
    mma_k8(d, a[1][0], a[1][1], b[1]);
    mma_k8(d, a[0][0], a[0][1], b[2]);
    mma_k8(d, a[1][0], a[1][1], b[0]);
    mma_k8(d, a[0][0], a[0][1], b[1]);
    mma_k8(d, a[0][0], a[0][1], b[0]);
}

template <int DH>
__global__ void __launch_bounds__(F6_THREADS, DH <= 40 ? 4 : DH <= 80 ? 2 : 1) spatial_attention_x6_kernel(const FlashArgs a) {
    using Cfg = F6Cfg<DH>;
    constexpr int PITCH = Cfg::PITCH, CH = Cfg::CH, NT = Cfg::NT, KS16 = Cfg::KS16, QTILE = Cfg::QTILE, KTILE = Cfg::KTILE;
    extern __shared__ __align__(128) uint8_t f6_smem[];
    pdl_wait();
    pdl_launch_dependents();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q0 = blockIdx.x * F6_BM, head = blockIdx.y, img = blockIdx.z;
    const bf16 *qg = (const bf16 *)a.q + (int64_t)img * a.q_bs + head * DH;
    const int kv_img = img / a.kv_div;
    const bf16 *kg = (const bf16 *)a.k + (int64_t)kv_img * a.kv_bs + head * DH;
    const bf16 *vg = (const bf16 *)a.v + (int64_t)kv_img * a.kv_bs + head * DH;
    const uint32_t sq = (uint32_t)__cvta_generic_to_shared(f6_smem);          // Q plane p at sq + p QTILE
    const uint32_t st0 = sq + 3 * QTILE;                                       // stage s: Kh Km Kl Vh Vm Vl at st0 + (6 s + {0..5}) KTILE
    const int Lq = a.Lq, Lkv = a.Lkv;

    for (int i = tid; i < F6_BM * CH; i += F6_THREADS) {
        const int r = i / CH, c = i - r * CH;
        const int row = q0 + r;
        const bool ok = row < Lq;
        const bf16 *src = qg + (int64_t)(ok ? row : Lq - 1) * a.q_rs + c * 8;
        const uint32_t so = (uint32_t)(r * PITCH + c * 8) * 2;
#pragma unroll
        for (int p = 0; p < 3; p++) f6_cp16(sq + p * QTILE + so, src + p * a.q_lo_off, ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    auto load_kv = [&](int t, int stage) {
        const uint32_t sb = st0 + stage * 6 * KTILE;
        for (int i = tid; i < F6_BN * CH; i += F6_THREADS) {
            const int r = i / CH, c = i - r * CH;
            const int key = t * F6_BN + r;
            const bool ok = key < Lkv;
            const int64_t off = (int64_t)(ok ? key : Lkv - 1) * a.kv_rs + c * 8;
            const uint32_t so = (uint32_t)(r * PITCH + c * 8) * 2;
#pragma unroll
            for (int p = 0; p < 3; p++) {
                f6_cp16(sb + p * KTILE + so, kg + off + p * a.kv_lo_off, ok);
                f6_cp16(sb + (3 + p) * KTILE + so, vg + off + p * a.kv_lo_off, ok);
            }
        }
    };
    load_kv(0, 0);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncthreads();

    const uint32_t qa = sq + (uint32_t)((warp * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * PITCH + 8 * (lane >> 4)) * 2;
    const uint32_t qa8 = sq + (uint32_t)((warp * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * PITCH) * 2 + KS16 * 32;
    uint32_t qf[Cfg::QRES ? KS16 : 1][3][4];
    uint32_t qt[3][2] = {{0u, 0u}, {0u, 0u}, {0u, 0u}};
    if constexpr (Cfg::QRES) {
#pragma unroll
        for (int ks = 0; ks < KS16; ks++)
#pragma unroll
            for (int p = 0; p < 3; p++) ldsm_x4(qa + p * QTILE + ks * 32, qf[ks][p][0], qf[ks][p][1], qf[ks][p][2], qf[ks][p][3]);
    }
    if constexpr (Cfg::TAIL8) {
#pragma unroll
        for (int p = 0; p < 3; p++) ldsm_x2(qa8 + p * QTILE, qt[p][0], qt[p][1]);
    }

    float o[NT][4];
#pragma unroll
    for (int n = 0; n < NT; n++) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    const float sc = a.scale;
    const int nt = (Lkv + F6_BN - 1) / F6_BN;
    const uint32_t k_lane = (uint32_t)((lane & 7) * PITCH + 8 * ((lane >> 3) & 1)) * 2;                       // x2: keys 8j.., channels 0-7 | 8-15 of a k16 step
    const uint32_t v_lane = (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * PITCH + 8 * (lane >> 4)) * 2;   // x4.trans: keys 0-7 | 8-15, channel tiles n | n + 1

    for (int t = 0; t < nt; t++) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        if (t + 1 < nt) load_kv(t + 1, (t + 1) & 1);
        asm volatile("cp.async.commit_group;" ::: "memory");
        const uint32_t sb = st0 + (t & 1) * 6 * KTILE;
        const uint32_t sk = sb + k_lane, sv = sb + 3 * KTILE + v_lane;

        // ---- S = the six plane products of Q and K (16 x 32 per warp), unscaled ----
        float s[4][4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
            const uint32_t ko = (uint32_t)(8 * j * PITCH) * 2;
#pragma unroll
            for (int ks = 0; ks < KS16; ks++) {
                uint32_t kb[3][2];
#pragma unroll
                for (int p = 0; p < 3; p++) ldsm_x2(sk + p * KTILE + ko + ks * 32, kb[p][0], kb[p][1]);
                if constexpr (Cfg::QRES) {
                    mma6_k16(s[j], qf[ks], kb);
                } else {
                    uint32_t qr[3][4];
#pragma unroll
                    for (int p = 0; p < 3; p++) ldsm_x4(qa + p * QTILE + ks * 32, qr[p][0], qr[p][1], qr[p][2], qr[p][3]);
                    mma6_k16(s[j], qr, kb);
                }
            }
            if constexpr (Cfg::TAIL8) {
                uint32_t kt[3];
#pragma unroll
                for (int p = 0; p < 3; p++) ldsm_x1(sk + p * KTILE + ko + KS16 * 32, kt[p]);
                mma6_k8(s[j], qt, kt);
            }
        }
        if ((t + 1) * F6_BN > Lkv) {
            const int kbase = t * F6_BN + 2 * (lane & 3);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                if (kbase + 8 * j >= Lkv) { s[j][0] = -INFINITY; s[j][2] = -INFINITY; }
                if (kbase + 8 * j + 1 >= Lkv) { s[j][1] = -INFINITY; s[j][3] = -INFINITY; }
            }
        }
        // ---- online softmax in fp32 (weights expf((s - m) * scale)); weights split into bf16 hi + mid + lo ----
        float mx0 = m0, mx1 = m1;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
            mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float al0 = expf((m0 - mx0) * sc), al1 = expf((m1 - mx1) * sc);      // m = -inf before the first tile: 0
        m0 = mx0; m1 = mx1;
        float r0 = 0.f, r1 = 0.f;
        uint32_t pw[4][2][3];                                                      // [key octet j][row crow | crow + 8][plane]
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const float e0 = expf((s[j][0] - mx0) * sc), e1 = expf((s[j][1] - mx0) * sc);
            const float e2 = expf((s[j][2] - mx1) * sc), e3 = expf((s[j][3] - mx1) * sc);
            r0 += e0 + e1; r1 += e2 + e3;
            split3_bf16x2(e0, e1, pw[j][0][0], pw[j][0][1], pw[j][0][2]);
            split3_bf16x2(e2, e3, pw[j][1][0], pw[j][1][1], pw[j][1][2]);
        }
        l0 = fmaf(l0, al0, r0); l1 = fmaf(l1, al1, r1);
        // ---- O = al O + the six plane products of P and V: each tile's products accumulate from zero in the MMA (12 steps), and the running O
        // takes them with one round-to-nearest fp32 fma -- the mma.sync fp32 accumulation is not round-to-nearest, and accumulating all keys
        // in it makes the error grow with the key count ----
        uint32_t pa[2][3][4];
#pragma unroll
        for (int kk = 0; kk < 2; kk++)
#pragma unroll
            for (int p = 0; p < 3; p++) {
                pa[kk][p][0] = pw[2 * kk][0][p]; pa[kk][p][1] = pw[2 * kk][1][p]; pa[kk][p][2] = pw[2 * kk + 1][0][p]; pa[kk][p][3] = pw[2 * kk + 1][1][p];
            }
        auto fold = [&](float (&d)[4], const float (&t)[4]) {
            d[0] = fmaf(d[0], al0, t[0]); d[1] = fmaf(d[1], al0, t[1]); d[2] = fmaf(d[2], al1, t[2]); d[3] = fmaf(d[3], al1, t[3]);
        };
#pragma unroll
        for (int n = 0; n + 2 <= NT; n += 2) {
            float t0[4] = {0.f, 0.f, 0.f, 0.f}, t1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int kk = 0; kk < 2; kk++) {
                const uint32_t vo = (uint32_t)(16 * kk * PITCH) * 2;
                uint32_t b0[3][2], b1[3][2];
#pragma unroll
                for (int p = 0; p < 3; p++) ldsm_x4_t(sv + p * KTILE + vo + n * 16, b0[p][0], b0[p][1], b1[p][0], b1[p][1]);
                mma6_k16(t0, pa[kk], b0);
                mma6_k16(t1, pa[kk], b1);
            }
            fold(o[n], t0);
            fold(o[n + 1], t1);
        }
        if constexpr (NT % 2 == 1) {
            float t0[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int kk = 0; kk < 2; kk++) {
                const uint32_t vo = (uint32_t)(16 * kk * PITCH) * 2;
                uint32_t b0[3][2];
#pragma unroll
                for (int p = 0; p < 3; p++) ldsm_x2_t(sv + p * KTILE + vo + (NT - 1) * 16, b0[p][0], b0[p][1]);
                mma6_k16(t0, pa[kk], b0);
            }
            fold(o[NT - 1], t0);
        }
    }
    // ---- O / l -> fp32 rows (each quad writes 32 contiguous bytes) ----
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.f / l0, i1 = 1.f / l1;
    const int crow = lane >> 2, ccol = (lane & 3) * 2;
    float *og = (float *)a.o + (int64_t)img * a.o_bs + head * DH;
    const int row0 = q0 + warp * 16 + crow, row1 = row0 + 8;
#pragma unroll
    for (int n = 0; n < NT; n++) {
        if (row0 < Lq) *reinterpret_cast<float2 *>(og + (int64_t)row0 * a.o_rs + 8 * n + ccol) = make_float2(o[n][0] * i0, o[n][1] * i0);
        if (row1 < Lq) *reinterpret_cast<float2 *>(og + (int64_t)row1 * a.o_rs + 8 * n + ccol) = make_float2(o[n][2] * i1, o[n][3] * i1);
    }
}

template <int DH>
static int launch_f6(const FlashArgs &a, cudaStream_t st) {
    using Cfg = F6Cfg<DH>;
    static DeviceOnce once;
    NMM_CUDA_OK(once.max_smem(spatial_attention_x6_kernel<DH>, Cfg::SMEM));
    const dim3 grid((unsigned)ceil_div(a.Lq, F6_BM), (unsigned)a.heads, (unsigned)a.images);
    const double per = (double)a.images * a.heads;
    ProfScope prof(K_SPATIAL_ATTN, st, 4.0 * per * a.Lq * (double)a.Lkv * DH, 4.0 * (2.0 * per * a.Lq * DH + 2.0 * per / a.kv_div * a.Lkv * DH));
    NMM_CUDA_OK(launch_pdl(spatial_attention_x6_kernel<DH>, grid, dim3(F6_THREADS), (size_t)Cfg::SMEM, st, a));
    NMM_LAUNCHED("spatial_attention_x6_kernel");
    return NMM_OK;
}

// q, k, v: bf16 hi | mid | lo planes (hi at the pointer, plane p `p * *_lo_off` elements further in the same row); o: fp32
int launch_spatial_attention_x6(const FlashArgs &a, cudaStream_t st) {
    if (a.Lq <= 0 || a.Lkv <= 0 || a.images <= 0 || a.heads <= 0 || a.kv_div <= 0) return fail(NMM_ERR_BAD_ARG, "spatial attention: non-positive size");
    if (a.images > 65535 || a.heads > 65535) return fail(NMM_ERR_UNSUPPORTED, "fp32-exact spatial attention: more than 65535 images or heads");
    if (!aligned(a.q, 16) || !aligned(a.k, 16) || !aligned(a.v, 16) || !aligned(a.o, 8) || a.q_rs % 8 || a.kv_rs % 8 || a.q_bs % 8 || a.kv_bs % 8 ||
        a.q_lo_off % 8 || a.kv_lo_off % 8 || a.o_rs % 2 || a.o_bs % 2)
        return fail(NMM_ERR_BAD_ARG, "fp32-exact spatial attention: misaligned operand planes");
    switch (a.dh) {
        case 40: return launch_f6<40>(a, st);
        case 80: return launch_f6<80>(a, st);
        case 160: return launch_f6<160>(a, st);
        default: break;
    }
    return fail(NMM_ERR_UNSUPPORTED, "fp32-exact spatial attention: head dim %d (supported: 40, 80, 160)", a.dh);
}

}  // namespace nmm

// Long-sequence attention of the UNet's spatial Transformer3DModel blocks (SURVEY 8(f) N3): per (image, head)
//     O = softmax(Q K^T * d_h^-1/2) V            Q: [Lq, d_h], K / V: [Lkv, d_h]
// for the self-attention over the h*w positions of one frame (Lq = Lkv = P <= 4096; animatediff/models/attention.py:277-280 -> the
// inherited CrossAttention.forward / _attention, motion_module_new.py:194-287) and the cross-attention onto the 77 text tokens
// (attention.py:282-292; Lkv = 77, the same K / V for every frame of a clip: `repeat(encoder_hidden_states, 'b n c -> (b f) n c')`,
// attention.py:101, is folded into the indexing -- kv image = q image / frames).
//
// Flash-style: the [Lq, Lkv] score matrix is never materialised (the reference writes + reads it: 8 heads x 4096^2 x 4 B = 537 MB per
// frame at the 64 x 64 level).  One CTA = 128 queries of one (image, head), 8 warps x 16 query rows; K / V stream through a
// double-buffered cp.async ring in 64-key tiles; S = Q K^T and O += P V on mma.sync m16n8k16 (bf16 -> fp32) with the Q fragments
// resident in registers, the online softmax (base 2, running max / sum per row) on the accumulator fragments in fp32, P fed back
// to the tensor core as bf16 straight from the S fragments.  Head split / merge (motion_module_new.py:181-193) is indexing: q, k, v
// are column slices [head * d_h, (head + 1) * d_h) of the projection outputs, O lands in the same slice of ctx.
// d_h in {40, 80, 160} (C / 8 at the UNet's widths): d_h = 40 runs its 2.5 k-steps as k16 + k16 + k8.
// Row pitch in shared memory: d_h (+ 8) elements so that pitch / 16 B is odd -> the 8 rows of an ldmatrix hit distinct banks.
// tcgen05 is not used here on purpose (yet): at d_h = 40 the kernel is bounded by the 128 x 64 exponentials per tile on the SFU
// (16 / clk / SM) as much as by the tensor pipe; see DESIGN.md section 8 for the measured rate and the next step.
#include "attention_core.cuh"
#include "common.cuh"

namespace nmm {

constexpr int FA_BN = 64;       // keys per compute tile (S fragment = 16 x 64 per warp)
constexpr int FA_ST = 128;      // keys per pipeline stage = two compute tiles per __syncthreads (barrier stalls were 11 % of issue slots at 64)

// WARPS = 8 (128 queries per CTA) for the self-attention, 4 (64 queries per CTA, twice the CTAs per SM) for short key sequences -- the
// 77-token text cross-attention is a single key stage per CTA and lives on latency hiding across CTAs, not on K / V reuse.
template <int DH, int WARPS = 8>
struct FaCfg {
    static constexpr int FA_BM = 16 * WARPS, FA_THREADS = 32 * WARPS;
    static constexpr int PITCH = ((DH / 8) % 2 == 1) ? DH : DH + 8;     // elements
    static constexpr int CH = DH / 8;                                   // 16-byte chunks per row
    static constexpr int Q_BYTES = FA_BM * PITCH * 2;
    static constexpr int KV_BYTES = FA_ST * PITCH * 2;
    static constexpr int STAGES = WARPS == 8 ? 2 : 1;                   // the 4-warp variant only ever sees one key stage (<= 128 keys)
    static constexpr int SMEM = Q_BYTES + 2 * STAGES * KV_BYTES;        // Q | K stages | V stages
    static constexpr int KS16 = DH / 16;                                // full k16 steps of S = Q K^T
    static constexpr bool TAIL8 = (DH % 16) == 8;
    static constexpr int NT = DH / 8;                                   // n8 tiles of O
};

__device__ __forceinline__ void cp_async16(uint32_t saddr, const void *g, bool valid) {
    const int sz = valid ? 16 : 0;      // src-size 0: the 16 bytes are zero-filled, nothing is read
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// 2^x on the SFU, one instruction (exp2f() adds a denormal-range rescue: FSETP + FMUL + FMUL per value); flush-to-zero is what a
// softmax weight below 2^-126 should do anyway.  ex2(-inf) = +0.
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int DH, int WARPS>
__global__ void __launch_bounds__(32 * WARPS, DH <= 80 ? 16 / WARPS : 8 / WARPS) spatial_attention_kernel(const FlashArgs a) {
    using Cfg = FaCfg<DH, WARPS>;
    constexpr int FA_BM = Cfg::FA_BM, FA_THREADS = Cfg::FA_THREADS;
    constexpr int PITCH = Cfg::PITCH, CH = Cfg::CH, NT = Cfg::NT, KS16 = Cfg::KS16;
    extern __shared__ __align__(128) uint8_t fa_smem[];
    pdl_wait();
    pdl_launch_dependents();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q0 = blockIdx.x * FA_BM, head = blockIdx.y, img = blockIdx.z;
    const bf16 *qg = (const bf16 *)a.q + (int64_t)img * a.q_bs + head * DH;
    const int kv_img = img / a.kv_div;
    const bf16 *kg = (const bf16 *)a.k + (int64_t)kv_img * a.kv_bs + head * DH;
    const bf16 *vg = (const bf16 *)a.v + (int64_t)kv_img * a.kv_bs + head * DH;
    const uint32_t sq = (uint32_t)__cvta_generic_to_shared(fa_smem);
    const uint32_t sk0 = sq + Cfg::Q_BYTES, sv0 = sk0 + Cfg::STAGES * Cfg::KV_BYTES;
    const int Lq = a.Lq, Lkv = a.Lkv;

    for (int i = tid; i < FA_BM * CH; i += FA_THREADS) {
        const int r = i / CH, c = i - r * CH;
        const int row = q0 + r;
        const bool ok = row < Lq;
        cp_async16(sq + (uint32_t)(r * PITCH + c * 8) * 2, qg + (int64_t)(ok ? row : Lq - 1) * a.q_rs + c * 8, ok);
    }
    cp_async_commit();
    auto load_kv = [&](int t, int stage) {
        const uint32_t sk = sk0 + stage * Cfg::KV_BYTES, sv = sv0 + stage * Cfg::KV_BYTES;
        for (int i = tid; i < FA_ST * CH; i += FA_THREADS) {
            const int r = i / CH, c = i - r * CH;
            const int key = t * FA_ST + r;
            const bool ok = key < Lkv;
            const int64_t off = (int64_t)(ok ? key : Lkv - 1) * a.kv_rs + c * 8;
            const uint32_t so = (uint32_t)(r * PITCH + c * 8) * 2;
            cp_async16(sk + so, kg + off, ok);
            cp_async16(sv + so, vg + off, ok);
        }
    };
    load_kv(0, 0);
    cp_async_commit();

    // Q fragments of this warp's 16 rows (resident for the whole kernel)
    cp_async_wait<1>();
    __syncthreads();
    uint32_t qf[KS16][4];
    uint32_t qt[2] = {0u, 0u};
    {
        const uint32_t qa = sq + (uint32_t)((warp * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * PITCH + 8 * (lane >> 4)) * 2;
#pragma unroll
        for (int ks = 0; ks < KS16; ks++) ldsm_x4(qa + ks * 32, qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
        if constexpr (Cfg::TAIL8) {
            const uint32_t qa2 = sq + (uint32_t)((warp * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * PITCH) * 2 + KS16 * 32;
            ldsm_x2(qa2, qt[0], qt[1]);
        }
    }

    float o[NT][4];
#pragma unroll
    for (int n = 0; n < NT; n++) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    const float sl = a.scale_log2e;
    const int nt = (Lkv + FA_ST - 1) / FA_ST;
    const uint32_t k_lane = (uint32_t)((lane & 7) * PITCH + 8 * (lane >> 3)) * 2;
    const uint32_t v_lane = (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * PITCH + 8 * (lane >> 4)) * 2;

    for (int t = 0; t < nt; t++) {
        cp_async_wait<0>();
        __syncthreads();                       // tile t landed for everyone; everyone is done with tile t - 1 (the other stage)
        if (t + 1 < nt) load_kv(t + 1, (t + 1) & 1);
        cp_async_commit();
#pragma unroll 1
        for (int half = 0; half < FA_ST / FA_BN; half++) {
        const int key0 = t * FA_ST + half * FA_BN;
        if (key0 >= Lkv) break;
        const uint32_t sk = sk0 + (t & 1) * Cfg::KV_BYTES + (uint32_t)(half * FA_BN * PITCH) * 2 + k_lane;
        const uint32_t sv = sv0 + (t & 1) * Cfg::KV_BYTES + (uint32_t)(half * FA_BN * PITCH) * 2 + v_lane;

        // ---- S = Q K^T (16 x 64 per warp) ----
        float s[8][4];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
            const uint32_t ka = sk + (uint32_t)(8 * j * PITCH) * 2;
#pragma unroll
            for (int k0 = 0; k0 + 32 <= DH; k0 += 32) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4(ka + k0 * 2, b0, b1, b2, b3);
                mma_k16(s[j], qf[k0 / 16][0], qf[k0 / 16][1], qf[k0 / 16][2], qf[k0 / 16][3], b0, b1);
                mma_k16(s[j], qf[k0 / 16 + 1][0], qf[k0 / 16 + 1][1], qf[k0 / 16 + 1][2], qf[k0 / 16 + 1][3], b2, b3);
            }
            constexpr int K1 = DH / 32 * 32;
            if constexpr (DH - K1 >= 16) {
                uint32_t b0, b1;
                ldsm_x2(ka + K1 * 2, b0, b1);
                mma_k16(s[j], qf[K1 / 16][0], qf[K1 / 16][1], qf[K1 / 16][2], qf[K1 / 16][3], b0, b1);
            }
            if constexpr (Cfg::TAIL8) {
                uint32_t b0;
                ldsm_x1(ka + KS16 * 32, b0);
                mma_k8(s[j], qt[0], qt[1], b0);
            }
        }
        if (key0 + FA_BN > Lkv) {      // keys past the end of a ragged last tile
            const int kbase = key0 + 2 * (lane & 3);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                if (kbase + 8 * j >= Lkv) { s[j][0] = -INFINITY; s[j][2] = -INFINITY; }
                if (kbase + 8 * j + 1 >= Lkv) { s[j][1] = -INFINITY; s[j][3] = -INFINITY; }
            }
        }
        // ---- online softmax (rows lane / 4 and lane / 4 + 8 of the warp's 16) ----
        float mx0 = m0, mx1 = m1;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
            mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float al0 = fast_exp2((m0 - mx0) * sl), al1 = fast_exp2((m1 - mx1) * sl);
        m0 = mx0; m1 = mx1;
        const float ms0 = mx0 * sl, ms1 = mx1 * sl;
        float r0 = 0.f, r1 = 0.f;
        uint32_t p[8][2];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const float e0 = fast_exp2(fmaf(s[j][0], sl, -ms0)), e1 = fast_exp2(fmaf(s[j][1], sl, -ms0));
            const float e2 = fast_exp2(fmaf(s[j][2], sl, -ms1)), e3 = fast_exp2(fmaf(s[j][3], sl, -ms1));
            p[j][0] = pack_bf16x2(e0, e1); p[j][1] = pack_bf16x2(e2, e3);
            // the row sum adds the ROUNDED weights: O / l is then an exact weighted mean with the weights the tensor core used
            r0 += bf16_lo(p[j][0]) + bf16_hi(p[j][0]); r1 += bf16_lo(p[j][1]) + bf16_hi(p[j][1]);
        }
        l0 = fmaf(l0, al0, r0); l1 = fmaf(l1, al1, r1);       // per-thread partial sums; the quad is reduced once at the end
#pragma unroll
        for (int n = 0; n < NT; n++) { o[n][0] *= al0; o[n][1] *= al0; o[n][2] *= al1; o[n][3] *= al1; }
        // ---- O += P V ----
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            const uint32_t va = sv + (uint32_t)(16 * kk * PITCH) * 2;
            const uint32_t a0 = p[2 * kk][0], a1 = p[2 * kk][1], a2 = p[2 * kk + 1][0], a3 = p[2 * kk + 1][1];
#pragma unroll
            for (int n = 0; n + 2 <= NT; n += 2) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4_t(va + n * 16, b0, b1, b2, b3);
                mma_k16(o[n], a0, a1, a2, a3, b0, b1);
                mma_k16(o[n + 1], a0, a1, a2, a3, b2, b3);
            }
            if constexpr (NT % 2 == 1) {
                uint32_t b0, b1;
                ldsm_x2_t(va + (NT - 1) * 16, b0, b1);
                mma_k16(o[NT - 1], a0, a1, a2, a3, b0, b1);
            }
        }
        }      // half
    }
    // ---- normalise, stage the warp's 16 x d_h block in its own (dead) Q rows, 16-byte stores ----
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.f / l0, i1 = 1.f / l1;
    const int crow = lane >> 2, ccol = (lane & 3) * 2;
    const uint32_t ob = sq + (uint32_t)((warp * 16 + crow) * PITCH + ccol) * 2;
    __syncwarp();
#pragma unroll
    for (int n = 0; n < NT; n++) {
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(ob + n * 16), "r"(pack_bf16x2(o[n][0] * i0, o[n][1] * i0)) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(ob + (uint32_t)(8 * PITCH) * 2 + n * 16), "r"(pack_bf16x2(o[n][2] * i1, o[n][3] * i1)) : "memory");
    }
    __syncwarp();
    bf16 *og = (bf16 *)a.o + (int64_t)img * a.o_bs + head * DH;
    for (int i = lane; i < 16 * CH; i += 32) {
        const int r = i / CH, c = i - r * CH;
        const int row = q0 + warp * 16 + r;
        if (row < Lq) {
            uint4 v;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sq + (uint32_t)((warp * 16 + r) * PITCH + c * 8) * 2));
            *reinterpret_cast<uint4 *>(og + (int64_t)row * a.o_rs + c * 8) = v;
        }
    }
}

// fp32 checker path (NMM_F32, small shapes): one warp per (query, head); lanes split the keys, fp32 throughout -- so that the fp32 parity
// mode of the spatial transformer has no bf16 rounding anywhere (bar 1e-4), like the FMA-pipe GEMM.  Large shapes run the tiled kernel of
// spatial_attention_f32.cu, which keeps this arithmetic.
template <int DH>
__global__ void __launch_bounds__(128) spatial_attention_f32_kernel(const float *__restrict__ q, const float *__restrict__ k, const float *__restrict__ v,
                                                                     float *__restrict__ o, int64_t q_rs, int64_t kv_rs, int64_t o_rs, int64_t q_bs,
                                                                     int64_t kv_bs, int64_t o_bs, int Lq, int Lkv, int kv_div, float scale) {
    pdl_wait();
    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 4 + warp, head = blockIdx.y, img = blockIdx.z;
    if (row >= Lq) return;
    const float *qp = q + (int64_t)img * q_bs + (int64_t)row * q_rs + head * DH;
    const float *kp = k + (int64_t)(img / kv_div) * kv_bs + head * DH;
    const float *vp = v + (int64_t)(img / kv_div) * kv_bs + head * DH;
    float qr[DH];
#pragma unroll
    for (int d = 0; d < DH; d++) qr[d] = qp[d] * scale;
    float m = -INFINITY, l = 0.f;
    float acc[DH];
#pragma unroll
    for (int d = 0; d < DH; d++) acc[d] = 0.f;
    for (int key = lane; key < Lkv; key += 32) {
        const float *kr = kp + (int64_t)key * kv_rs;
        float sc = 0.f;
#pragma unroll
        for (int d = 0; d < DH; d++) sc = fmaf(qr[d], kr[d], sc);
        const float mn = fmaxf(m, sc);
        const float al = expf(m - mn), e = expf(sc - mn);
        m = mn;
        l = l * al + e;
        const float *vr = vp + (int64_t)key * kv_rs;
#pragma unroll
        for (int d = 0; d < DH; d++) acc[d] = fmaf(acc[d], al, e * vr[d]);
    }
    // merge the 32 lanes' partial softmaxes
    const float mall = warp_max(m);
    const float f = (m == -INFINITY) ? 0.f : expf(m - mall);
    l = warp_sum(l * f);
    float *op = o + (int64_t)img * o_bs + (int64_t)row * o_rs + head * DH;
#pragma unroll
    for (int d = 0; d < DH; d++) {
        const float t = warp_sum(acc[d] * f);
        if (lane == (d & 31)) op[d] = t / l;
    }
}

template <int DH, int WARPS>
static int launch_flash_w(const FlashArgs &a, cudaStream_t st) {
    using Cfg = FaCfg<DH, WARPS>;
    static DeviceOnce once;
    NMM_CUDA_OK(once.max_smem(spatial_attention_kernel<DH, WARPS>, Cfg::SMEM));
    const dim3 grid((unsigned)ceil_div(a.Lq, Cfg::FA_BM), (unsigned)a.heads, (unsigned)a.images);
    const double per = (double)a.images * a.heads;
    ProfScope prof(K_SPATIAL_ATTN, st, 4.0 * per * a.Lq * (double)a.Lkv * DH,
                   2.0 * (2.0 * per * a.Lq * DH + 2.0 * per / a.kv_div * a.Lkv * DH));
    NMM_CUDA_OK(launch_pdl(spatial_attention_kernel<DH, WARPS>, grid, dim3(Cfg::FA_THREADS), (size_t)Cfg::SMEM, st, a));
    NMM_LAUNCHED("spatial_attention_kernel");
    return NMM_OK;
}

template <int DH>
static int launch_flash_t(const FlashArgs &a, cudaStream_t st) {
    // one key stage (<= 128 keys: the text cross-attention) and enough queries to fill the GPU with the smaller CTAs
    if (a.Lkv <= FA_ST && opt(NMM_OPT_SPATIAL_ATTN) != 25) return launch_flash_w<DH, 4>(a, st);
    return launch_flash_w<DH, 8>(a, st);
}

template <int DH>
static int launch_flash_f32_t(const FlashArgs &a, cudaStream_t st) {
    const dim3 grid((unsigned)ceil_div(a.Lq, 4), (unsigned)a.heads, (unsigned)a.images);
    const double per = (double)a.images * a.heads;
    ProfScope prof(K_SPATIAL_ATTN, st, 4.0 * per * a.Lq * (double)a.Lkv * DH, 4.0 * (2.0 * per * a.Lq * DH + 2.0 * per / a.kv_div * a.Lkv * DH));
    NMM_CUDA_OK(launch_pdl(spatial_attention_f32_kernel<DH>, grid, dim3(128), (size_t)0, st, (const float *)a.q, (const float *)a.k, (const float *)a.v,
                           (float *)a.o, a.q_rs, a.kv_rs, a.o_rs, a.q_bs, a.kv_bs, a.o_bs, a.Lq, a.Lkv, a.kv_div, a.scale));
    NMM_LAUNCHED("spatial_attention_f32_kernel");
    return NMM_OK;
}

int launch_spatial_attention(const FlashArgs &a, cudaStream_t st) {
    if (a.Lq <= 0 || a.Lkv <= 0 || a.images <= 0 || a.heads <= 0 || a.kv_div <= 0) return fail(NMM_ERR_BAD_ARG, "spatial attention: non-positive size");
    if (a.images > 65535 || a.heads > 65535) return fail(NMM_ERR_UNSUPPORTED, "spatial attention: more than 65535 images / heads");
    const int variant = (int)opt(NMM_OPT_SPATIAL_ATTN);
    if (variant != 1 && spatial_attention_tc_eligible(a)) return launch_spatial_attention_tc(a, variant, st);
    if (a.dtype == NMM_BF16) {
        if (!aligned(a.q, 16) || !aligned(a.k, 16) || !aligned(a.v, 16) || !aligned(a.o, 16) || a.q_rs % 8 || a.kv_rs % 8 || a.o_rs % 8 || a.q_bs % 8 ||
            a.kv_bs % 8 || a.o_bs % 8)
            return fail(NMM_ERR_BAD_ARG, "spatial attention: q / k / v / o must be 16-byte aligned with strides in multiples of 8 elements");
        switch (a.dh) {
            case 40: return launch_flash_t<40>(a, st);
            case 80: return launch_flash_t<80>(a, st);
            case 160: return launch_flash_t<160>(a, st);
            default: break;
        }
    } else if (a.dtype == NMM_F32) {
        // Two kernels with the same arithmetic: the tiled flash kernel on the FMA pipe (spatial_attention_f32.cu) from F32_TILED_MIN_SCORES
        // score elements up, the checker (one warp per query, keys streamed from L2) below.  Measured on B200 the tiled kernel is the faster
        // one at every swept size, from 8e3 score elements up (1.5-4x at 1e4-1e5, 45-65x from 1e7; profiles/r3_spatial_fp32_attention.txt).
        // The checker is kept below 2^17, where a call costs 0.02-0.26 ms either way, so that small fp32 calls (the parity fixtures, the
        // tests) keep the results of earlier releases bit for bit.
        constexpr double F32_TILED_MIN_SCORES = 1 << 17;
        const double scores = (double)a.Lq * a.Lkv * a.images * a.heads;
        const bool tiled = spatial_attention_f32_tiled_eligible(a);
        if (variant == 30 && !tiled) return fail(NMM_ERR_BAD_ARG, "fp32 tiled spatial attention needs 16-byte aligned q / k / v with strides in multiples of 4");
        if (tiled && variant != 31 && (variant == 30 || scores >= F32_TILED_MIN_SCORES)) return launch_spatial_attention_f32_tiled(a, st);
        // the checker takes minutes at the 64 x 64 level: refuse misaligned operands there instead of appearing to hang
        if (variant != 31 && scores > 1.1e9)
            return fail(NMM_ERR_UNSUPPORTED, "fp32 spatial attention of %d x %d keys x %d images x %d heads needs 16-byte aligned q / k / v with "
                        "strides in multiples of 4 (the tiled kernel)", a.Lq, a.Lkv, a.images, a.heads);
        switch (a.dh) {
            case 40: return launch_flash_f32_t<40>(a, st);
            case 80: return launch_flash_f32_t<80>(a, st);
            case 160: return launch_flash_f32_t<160>(a, st);
            default: break;
        }
    }
    return fail(NMM_ERR_UNSUPPORTED, "spatial attention: head dim %d / dtype %d not supported (d_h in {40, 80, 160}; bf16 or fp32)", a.dh, a.dtype);
}

}  // namespace nmm

// Short-sequence temporal self-attention: softmax(q k^T * d_h^-1/2) v over the frame axis (F <= 32),
// independently per (batch, spatial position, head).
//
// Reference arithmetic: CrossAttention._attention, motion_module_new.py:258-287 (baddbmm(beta=0, alpha=scale)
// -> softmax(dim=-1) -> bmm), with reshape_heads_to_batch_dim / reshape_batch_dim_to_heads (:181-193) and the
// "(b f) d c -> (b d) f c" / inverse rearranges of VersatileAttention.forward (motion_module.py:275,327) folded
// into the addressing: a token row is n = (b*F + f)*P + p, so the F rows of one position are P rows apart.
//
// Mapping: one thread per (position, head, query frame).  A CTA stages the q|k|v rows of PB consecutive
// positions x all F frames in shared memory with 16-byte coalesced loads (each frame contributes one
// contiguous PB*3C-element run), keeps the F scores in registers, does the softmax in fp32 and writes its
// context row back through shared memory so the global stores are 16-byte coalesced as well.
// HBM-bound: bytes = 4*N*C*s (read qkv, write ctx), flops = 4*N*F*C.
#include <cstdlib>

#include "common.cuh"
#include "attention_core.cuh"

namespace nmm {

template <typename T, int VEC> struct RowVec;
template <> struct RowVec<bf16, 8> {
    static __device__ __forceinline__ void load(const bf16 *p, float (&f)[8]) {
        uint4 v = *reinterpret_cast<const uint4 *>(p);
        f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
        f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
    }
    static __device__ __forceinline__ void store(bf16 *p, const float (&f)[8]) {
        *reinterpret_cast<uint4 *>(p) = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]),
                                                   pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
    }
};
template <> struct RowVec<float, 4> {
    static __device__ __forceinline__ void load(const float *p, float (&f)[4]) {
        float4 v = *reinterpret_cast<const float4 *>(p);
        f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
    }
    static __device__ __forceinline__ void store(float *p, const float (&f)[4]) {
        *reinterpret_cast<float4 *>(p) = make_float4(f[0], f[1], f[2], f[3]);
    }
};
template <typename T> struct RowVec<T, 1> {
    static __device__ __forceinline__ void load(const T *p, float (&f)[1]) { f[0] = to_f32(*p); }
    static __device__ __forceinline__ void store(T *p, const float (&f)[1]) { *p = from_f32<T>(f[0]); }
};

// A CTA handles PB positions x HB heads (blockIdx.y selects the head group; HB == heads for the UNet's 320/640-channel
// levels, fewer for 1280 channels so the tile fits shared memory).
// smem layout: [PB positions][F frames][q(HB*dh) | k(HB*dh) | v(HB*dh) | PAD] elements of T; PAD keeps consecutive frame
// rows on different banks (row pitch in bytes = 3*HB*dh*s + 16).
template <typename T, int VEC, int FMAX>
__global__ void __launch_bounds__(256) temporal_attention_kernel(const T *__restrict__ qkv, T *__restrict__ ctx, int B, int F,
                                                                 int P, int C, int heads, int PB, int HB, float scale, int split_out) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sm = reinterpret_cast<T *>(smem_raw);
    constexpr int PAD = 16 / (int)sizeof(T);
    const int dh = C / heads;
    const int W = HB * dh;                      // channels of this head group
    const int c_off = blockIdx.y * W;           // first channel of the head group
    const int pitch = 3 * W + PAD;
    const int tiles_per_img = (P + PB - 1) / PB;
    const int b = blockIdx.x / tiles_per_img;
    const int p0 = (blockIdx.x % tiles_per_img) * PB;
    const int npos = min(PB, P - p0);
    const int tid = threadIdx.x, nthr = blockDim.x;

    // ---- stage q|k|v with cp.async (16-byte LDGSTS, no register staging): one warp per (frame, position) row at a time,
    //      lanes striding over the row's vectors; the three segments (q, k, v of this head group) are W elements each --------
    {
        constexpr int LV = 16 / (int)sizeof(T);                     // elements per 16-byte copy
        const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
        const int rows = F * npos;
        if (VEC > 1) {                                              // host guarantees 16-byte alignment when VEC > 1
            const int vec_per_seg = W / LV;
            for (int r = warp; r < rows; r += nwarps) {
                const int f = r / npos, pl = r - f * npos;
                const T *src_row = qkv + ((int64_t)(b * F + f) * P + p0 + pl) * (3 * C) + c_off;
                const uint32_t dst_row = (uint32_t)__cvta_generic_to_shared(sm + (pl * F + f) * pitch);
#pragma unroll
                for (int seg = 0; seg < 3; seg++)
                    for (int v = lane; v < vec_per_seg; v += 32)
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_row + (uint32_t)((seg * W + v * LV) * sizeof(T))),
                                     "l"(src_row + seg * C + v * LV)
                                     : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        } else {
            for (int r = warp; r < rows; r += nwarps) {
                const int f = r / npos, pl = r - f * npos;
                const T *src_row = qkv + ((int64_t)(b * F + f) * P + p0 + pl) * (3 * C) + c_off;
                T *dst_row = sm + (pl * F + f) * pitch;
                for (int seg = 0; seg < 3; seg++)
                    for (int e = lane; e < W; e += 32) dst_row[seg * W + e] = src_row[seg * C + e];
            }
        }
    }
    __syncthreads();

    // ---- one thread per (pl, head, f) ---------------------------------------------------------------
    const int per_pos = HB * F;
    const int pl = tid / per_pos;
    const int hf = tid % per_pos;
    const int head = hf / F, f = hf % F;
    const bool active = pl < npos;             // tid < PB*heads*F by launch configuration
    if (active) {
        T *qrow = sm + (pl * F + f) * pitch + head * dh;             // this thread's query row (reused for output)
        const T *kbase = sm + (pl * F) * pitch + W + head * dh;
        const T *vbase = sm + (pl * F) * pitch + 2 * W + head * dh;
        float sc[FMAX];
#pragma unroll
        for (int j = 0; j < FMAX; j++) sc[j] = 0.f;
        for (int d = 0; d < dh; d += VEC) {
            float q[VEC];
            RowVec<T, VEC>::load(qrow + d, q);
#pragma unroll
            for (int j = 0; j < FMAX; j++) {
                if (j < F) {
                    float k[VEC];
                    RowVec<T, VEC>::load(kbase + j * pitch + d, k);
#pragma unroll
                    for (int e = 0; e < VEC; e++) sc[j] = fmaf(q[e], k[e], sc[j]);
                }
            }
        }
        // softmax over the F keys (fp32; the reference computes it in the input dtype -- fp32 as shipped)
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < FMAX; j++) if (j < F) { sc[j] *= scale; mx = fmaxf(mx, sc[j]); }
        float den = 0.f;
#pragma unroll
        for (int j = 0; j < FMAX; j++) if (j < F) { sc[j] = __expf(sc[j] - mx); den += sc[j]; }
        const float inv = 1.0f / den;
#pragma unroll
        for (int j = 0; j < FMAX; j++) if (j < F) sc[j] *= inv;
        for (int d = 0; d < dh; d += VEC) {
            float o[VEC];
#pragma unroll
            for (int e = 0; e < VEC; e++) o[e] = 0.f;
#pragma unroll
            for (int j = 0; j < FMAX; j++) {
                if (j < F) {
                    float v[VEC];
                    RowVec<T, VEC>::load(vbase + j * pitch + d, v);
#pragma unroll
                    for (int e = 0; e < VEC; e++) o[e] = fmaf(sc[j], v[e], o[e]);
                }
            }
            RowVec<T, VEC>::store(qrow + d, o);                       // q slot is private to this thread
        }
    }
    __syncthreads();

    // ---- write ctx rows (the first W elements of each staged row): one warp per row, 16-byte coalesced stores ----------
    {
        constexpr int LV = 16 / (int)sizeof(T);
        const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
        const int rows = F * npos;
        for (int r = warp; r < rows; r += nwarps) {
            const int f2 = r / npos, pl2 = r - f2 * npos;
            const T *src_row = sm + (pl2 * F + f2) * pitch;
            if constexpr (sizeof(T) == 4) {
                if (split_out) {                      // NMM_F32X3 / X6: ctx is the next GEMM's A operand, bf16 [N, 2C / 3C] hi | lo (| mid | lo) planes
                    bf16 *srow = reinterpret_cast<bf16 *>(ctx) + ((int64_t)(b * F + f2) * P + p0 + pl2) * (split_out * C);
                    if (VEC > 1) {
                        for (int v = lane; v < W / 4; v += 32) {
                            const float4 f4 = *reinterpret_cast<const float4 *>(src_row + v * 4);
                            if (split_out == 3) split4_store<3>(srow, C, c_off + v * 4, f4.x, f4.y, f4.z, f4.w);
                            else split4_store(srow, C, c_off + v * 4, f4.x, f4.y, f4.z, f4.w);
                        }
                    } else {
                        for (int e = lane; e < W; e += 32) {
                            if (split_out == 3) split1_store<3>(srow, C, c_off + e, to_f32(src_row[e]));
                            else split1_store(srow, C, c_off + e, to_f32(src_row[e]));
                        }
                    }
                    continue;
                }
            }
            T *dst_row = ctx + ((int64_t)(b * F + f2) * P + p0 + pl2) * C + c_off;
            if (VEC > 1) {
                for (int v = lane; v < W / LV; v += 32)
                    *reinterpret_cast<uint4 *>(dst_row + v * LV) = *reinterpret_cast<const uint4 *>(src_row + v * LV);
            } else {
                for (int e = lane; e < W; e += 32) dst_row[e] = src_row[e];
            }
        }
    }
}

template <typename T, int VEC>
static int launch_attn_t(const Geo &g, const T *qkv, T *ctx, cudaStream_t st, int split_out = 0) {
    if (g.heads * g.F > 256 && g.F > 256) return fail(NMM_ERR_UNSUPPORTED, "frames too large");
    const size_t smem_cap = 200 * 1024, smem_pref = 32 * 1024;       // <= 32 KB: ~7 CTAs per SM, so load / compute / store phases of different CTAs overlap
    auto row_bytes = [&](int hb) { return (size_t)(3 * hb * g.dh) * sizeof(T) + 16; };
    // heads per CTA: the largest divisor of `heads` whose tile fits the preferred budget, else the largest that fits at all
    int HB = 0, PB = 1;
    for (int pass = 0; pass < 2 && HB == 0; pass++) {
        const size_t budget = pass == 0 ? smem_pref : smem_cap;
        for (int hb = g.heads; hb >= 1; hb--) {
            if (g.heads % hb || hb * g.F > 256) continue;
            int pb = 256 / (hb * g.F);
            if (pb > g.P) pb = g.P;
            while (pb > 1 && (size_t)pb * g.F * row_bytes(hb) > budget) pb--;
            if ((size_t)pb * g.F * row_bytes(hb) <= budget) { HB = hb; PB = pb; break; }
        }
    }
    if (HB == 0) return fail(NMM_ERR_UNSUPPORTED, "attention tile does not fit shared memory (C=%d, F=%d)", g.C, g.F);
    const int per_pos = HB * g.F;
    const size_t smem = (size_t)PB * g.F * row_bytes(HB);
    const int threads = ((PB * per_pos + 31) / 32) * 32;
    const int64_t blocks = (int64_t)g.B * ceil_div(g.P, PB);
    if (blocks > 0x7fffffff) return fail(NMM_ERR_UNSUPPORTED, "attention grid too large");
    const dim3 grid((unsigned)blocks, (unsigned)(g.heads / HB));
    const float scale = 1.0f / sqrtf((float)g.dh);
#define ATTN_CASE(FM)                                                                                                    \
    do {                                                                                                                 \
        auto kern = temporal_attention_kernel<T, VEC, FM>;                                                               \
        static DeviceOnce once; /* per instantiation and device; never inside a stream capture after warm-up */            \
        NMM_CUDA_OK(once.max_smem(kern, (int)smem_cap));          \
        ProfScope prof(K_ATTENTION, st, 4.0 * g.N * g.F * g.C, 4.0 * g.N * g.C * sizeof(T));                             \
        launch_pdl(kern, grid, threads, smem, st, qkv, ctx, g.B, g.F, g.P, g.C, g.heads, PB, HB, scale, split_out);                          \
    } while (0)
    if (g.F <= 8) ATTN_CASE(8);
    else if (g.F <= 16) ATTN_CASE(16);
    else ATTN_CASE(32);
#undef ATTN_CASE
    NMM_LAUNCHED("temporal_attention_kernel");
    return NMM_OK;
}


// ------------------------------------------------------------------------------------------------------------------------
// Tensor-core variant for the shapes NEURONS actually runs (bf16, F = 8 or 16 frames, d_h % 8 == 0).
// One warp per (position, head) problem: S = Q K^T and O = P V on mma.sync (m16n8k16 / m16n8k8 bf16 -> fp32).  These are
// F x F x d_h problems (8 x 8 x 40 ...): far below the 64-row minimum of tcgen05, so the warp-level MMA is the right tool;
// it replaces ~1500 scalar instructions per thread of the SIMT kernel with ~20 MMAs + ~25 ldmatrix per warp.
// Staging, head-group tiling and the coalesced write-back are shared with the SIMT kernel above.
// The probabilities are fed to the second MMA as a bf16 hi + lo pair (two MMAs), so P carries ~16 mantissa bits.
// ------------------------------------------------------------------------------------------------------------------------
template <int F>      // 8 or 16
__global__ void __launch_bounds__(256) temporal_attention_mma_kernel(const bf16 *__restrict__ qkv, bf16 *__restrict__ ctx, int B, int P,
                                                                     int C, int heads, int PB, int HB, float scale_log2e) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    extern __shared__ __align__(16) unsigned char smem_raw[];
    bf16 *sm = reinterpret_cast<bf16 *>(smem_raw);
    constexpr int PAD = 8;
    constexpr int NT = F / 8;                   // key tiles of 8
    const int dh = C / heads;
    const int W = HB * dh;
    const int c_off = blockIdx.y * W;
    const int pitch = 3 * W + PAD;              // elements; (pitch*2/4) % 32 == 4 for W % 64 == 0: ldmatrix rows hit distinct banks
    const int tiles_per_img = (P + PB - 1) / PB;
    const int b = blockIdx.x / tiles_per_img;
    const int p0 = (blockIdx.x % tiles_per_img) * PB;
    const int npos = min(PB, P - p0);
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
    const int rows = F * npos;

    // ---- stage q|k|v rows with cp.async (same layout as the SIMT kernel) ------------------------------------------------
    {
        const int vec_per_seg = W / 8;
        for (int r = warp; r < rows; r += nwarps) {
            const int f = r / npos, pl = r - f * npos;
            const bf16 *src_row = qkv + ((int64_t)(b * F + f) * P + p0 + pl) * (3 * C) + c_off;
            const uint32_t dst_row = (uint32_t)__cvta_generic_to_shared(sm + (pl * F + f) * pitch);
#pragma unroll
            for (int seg = 0; seg < 3; seg++)
                for (int v = lane; v < vec_per_seg; v += 32)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_row + (uint32_t)((seg * W + v * 8) * 2)), "l"(src_row + seg * C + v * 8)
                                 : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();

    // ---- one warp per (position, head) ------------------------------------------------------------------------------------
    const uint32_t sm_u32 = (uint32_t)__cvta_generic_to_shared(sm);
    const int lrow = lane & 7, lmat = lane >> 3;          // ldmatrix: lanes 8m..8m+7 address the rows of matrix m
    const int crow = lane >> 2, ccol = (lane & 3) * 2;     // accumulator fragment: row crow (and crow + 8), columns ccol, ccol + 1
    for (int prob = warp; prob < npos * HB; prob += nwarps) {
        const int pl = prob / HB, hd = prob - pl * HB;
        const uint32_t qb = sm_u32 + (uint32_t)(((pl * F) * pitch + hd * dh) * 2);     // row f at + f * pitch * 2 bytes
        const uint32_t kb = qb + (uint32_t)(W * 2), vb = qb + (uint32_t)(2 * W * 2);
        const uint32_t rstride = (uint32_t)(pitch * 2);
        float s[NT][4];
#pragma unroll
        for (int j = 0; j < NT; j++) { s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f; }
        // S = Q K^T over d in steps of 16 (+ one step of 8 when d_h % 16 == 8)
        int k0 = 0;
        for (; k0 + 16 <= dh; k0 += 16) {
            uint32_t a0, a1 = 0u, a2, a3 = 0u;
            if constexpr (F == 16) {
                // matrices: (rows 0-7, k0), (rows 8-15, k0), (rows 0-7, k0+8), (rows 8-15, k0+8)
                ldsm_x4(qb + (uint32_t)(lrow + 8 * (lmat & 1)) * rstride + (uint32_t)((k0 + 8 * (lmat >> 1)) * 2), a0, a1, a2, a3);
            } else {
                ldsm_x2(qb + (uint32_t)lrow * rstride + (uint32_t)((k0 + 8 * (lmat & 1)) * 2), a0, a2);   // rows 8-15 are padding
            }
#pragma unroll
            for (int j = 0; j < NT; j++) {
                uint32_t b0, b1;
                ldsm_x2(kb + (uint32_t)(8 * j + lrow) * rstride + (uint32_t)((k0 + 8 * (lmat & 1)) * 2), b0, b1);
                mma_k16(s[j], a0, a1, a2, a3, b0, b1);
            }
        }
        if (k0 < dh) {      // 8 remaining columns
            uint32_t a0, a1 = 0u;
            if constexpr (F == 16) ldsm_x2(qb + (uint32_t)(lrow + 8 * (lmat & 1)) * rstride + (uint32_t)(k0 * 2), a0, a1);
            else ldsm_x1(qb + (uint32_t)lrow * rstride + (uint32_t)(k0 * 2), a0);
#pragma unroll
            for (int j = 0; j < NT; j++) {
                uint32_t b0;
                ldsm_x1(kb + (uint32_t)(8 * j + lrow) * rstride + (uint32_t)(k0 * 2), b0);
                mma_k8(s[j], a0, a1, b0);
            }
        }
        // softmax over the keys of row crow (regs 0,1) and row crow + 8 (regs 2,3; F == 16 only), fp32, base-2 exponentials
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int j = 0; j < NT; j++) { mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1])); mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3])); }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
        for (int j = 0; j < NT; j++) {
            s[j][0] = exp2f((s[j][0] - mx0) * scale_log2e); s[j][1] = exp2f((s[j][1] - mx0) * scale_log2e);
            sum0 += s[j][0] + s[j][1];
            if constexpr (F == 16) {
                s[j][2] = exp2f((s[j][2] - mx1) * scale_log2e); s[j][3] = exp2f((s[j][3] - mx1) * scale_log2e);
                sum1 += s[j][2] + s[j][3];
            }
        }
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
        const float inv0 = 1.0f / sum0, inv1 = (F == 16) ? 1.0f / sum1 : 0.f;
        // P as the A operand of the second MMA (accumulator layout == A layout for these shapes), bf16 hi + lo
        uint32_t ph[4] = {0u, 0u, 0u, 0u}, pl_[4] = {0u, 0u, 0u, 0u};
        split_bf16x2(s[0][0] * inv0, s[0][1] * inv0, ph[0], pl_[0]);                       // row crow, keys 0-7
        if constexpr (F == 16) {
            split_bf16x2(s[0][2] * inv1, s[0][3] * inv1, ph[1], pl_[1]);                   // row crow + 8, keys 0-7
            split_bf16x2(s[1][0] * inv0, s[1][1] * inv0, ph[2], pl_[2]);                   // row crow, keys 8-15
            split_bf16x2(s[1][2] * inv1, s[1][3] * inv1, ph[3], pl_[3]);                   // row crow + 8, keys 8-15
        }
        __syncwarp();                                   // all of this warp's reads of the q rows are done: reuse them for O
        // O = P V, 8 output columns per MMA
        for (int n0 = 0; n0 < dh; n0 += 8) {
            float o[4] = {0.f, 0.f, 0.f, 0.f};
            if constexpr (F == 16) {
                uint32_t b0, b1;
                ldsm_x2_t(vb + (uint32_t)(lrow + 8 * (lmat & 1)) * rstride + (uint32_t)(n0 * 2), b0, b1);   // keys 0-7, keys 8-15
                mma_k16(o, ph[0], ph[1], ph[2], ph[3], b0, b1);
                mma_k16(o, pl_[0], pl_[1], pl_[2], pl_[3], b0, b1);
            } else {
                uint32_t b0;
                ldsm_x1_t(vb + (uint32_t)lrow * rstride + (uint32_t)(n0 * 2), b0);
                mma_k8(o, ph[0], 0u, b0);
                mma_k8(o, pl_[0], 0u, b0);
            }
            // context row crow (and crow + 8) into the q slot of this problem
            bf16 *orow = sm + ((pl * F) + crow) * pitch + hd * dh + n0 + ccol;
            *reinterpret_cast<uint32_t *>(orow) = pack_bf16x2(o[0], o[1]);
            if constexpr (F == 16) *reinterpret_cast<uint32_t *>(orow + 8 * pitch) = pack_bf16x2(o[2], o[3]);
        }
    }
    __syncthreads();

    // ---- write ctx rows: one warp per row, 16-byte coalesced stores --------------------------------------------------------
    for (int r = warp; r < rows; r += nwarps) {
        const int f2 = r / npos, pl2 = r - f2 * npos;
        const bf16 *src_row = sm + (pl2 * F + f2) * pitch;
        bf16 *dst_row = ctx + ((int64_t)(b * F + f2) * P + p0 + pl2) * C + c_off;
        for (int v = lane; v < W / 8; v += 32)
            *reinterpret_cast<uint4 *>(dst_row + v * 8) = *reinterpret_cast<const uint4 *>(src_row + v * 8);
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// Compile-time specialisation of the kernel above for the head sizes of the SD1.5 levels (d_h = 40 / 80 / 160 with 8 heads):
// the head group is always W = 320 channels wide (8, 4 or 2 heads), so pitch, row offsets and every loop bound are constants.
// The runtime-shaped kernel spends ~580 warp instructions per (position, head) problem, >50 % of them integer address
// arithmetic (ncu: issue slots 81 % busy, ALU pipe 52 %, DRAM 52 %) -- i.e. it is issue-bound, not HBM-bound.  Here every
// ldmatrix / st.shared address is base + immediate, the loops are fully unrolled and staging / write-back use a flat chunk
// index, which removes most of that overhead.
// ------------------------------------------------------------------------------------------------------------------------
template <int F, int DH>      // F in {8, 16}; DH in {40, 80, 160}
__global__ void __launch_bounds__(256) temporal_attention_mma_fixed_kernel(const bf16 *__restrict__ qkv, bf16 *__restrict__ ctx, int P, int C,
                                                                           int PB, float scale_log2e) {
    pdl_wait();
    pdl_launch_dependents();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    bf16 *sm = reinterpret_cast<bf16 *>(smem_raw);
    constexpr int W = 320;
    constexpr int PITCH = 3 * W + 8;            // elements; 1936 B per row: (1936 / 4) % 32 == 4 -> ldmatrix rows hit distinct banks
    constexpr uint32_t RS = PITCH * 2;          // row stride in bytes
    const int c_off = blockIdx.y * W;
    const int tiles_per_img = (P + PB - 1) / PB;
    const int b = blockIdx.x / tiles_per_img;
    const int p0 = (blockIdx.x - b * tiles_per_img) * PB;
    const int npos = min(PB, P - p0);
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthr >> 5;
    const int rows = F * npos;                  // smem row r = pl * F + f
    const uint32_t sm_u32 = (uint32_t)__cvta_generic_to_shared(sm);

    {
        // ---- stage q|k|v rows: one warp per row, 120 16-byte chunks = 4 cp.async per lane (the last with 24 lanes) ------------
        // chunk w of a row lives at src_row + w * 8 + seg * (C - 320) elements, seg = w / 40 (the q | k | v segment)
        const bf16 *src0 = qkv + ((int64_t)b * F * P + p0) * (3 * (int64_t)C) + c_off;
        const uint32_t row_elems = 3u * (uint32_t)C, seg_skip = (uint32_t)(C - W);
        for (uint32_t r = warp; r < (uint32_t)rows; r += nwarps) {
            const uint32_t pl = r / F, f = r % F;                                     // F is a power of two
            const bf16 *srow = src0 + (f * (uint32_t)P + pl) * row_elems + lane * 8;   // element offset < 2^31: checked by the launcher
            const uint32_t drow = sm_u32 + r * RS + lane * 16;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (k < 3 || lane < 24) {
                    const uint32_t seg = k == 0 ? 0u : k == 1 ? (lane >= 8 ? 1u : 0u) : k == 2 ? (lane >= 16 ? 2u : 1u) : 2u;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(drow + k * 512), "l"(srow + k * 256 + seg * seg_skip) : "memory");
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
    }

    attention_tile_mma<F, DH, W>(sm_u32, npos, warp, nwarps, lane, scale_log2e);
    {
        __syncthreads();
        // ---- write ctx rows: one warp per row, 40 16-byte chunks (lanes 0-31, then lanes 0-7) ----------------------------------
        bf16 *dst0 = ctx + ((int64_t)b * F * P + p0) * (int64_t)C + c_off;
        for (uint32_t r = warp; r < (uint32_t)rows; r += nwarps) {
            const uint32_t pl = r / F, f = r % F;
            const bf16 *srow = sm + r * PITCH + lane * 8;
            bf16 *drow = dst0 + (f * (uint32_t)P + pl) * (uint32_t)C + lane * 8;
            const uint4 v0 = *reinterpret_cast<const uint4 *>(srow);
            uint4 v1 = make_uint4(0u, 0u, 0u, 0u);
            if (lane < 8) v1 = *reinterpret_cast<const uint4 *>(srow + 256);
            *reinterpret_cast<uint4 *>(drow) = v0;
            if (lane < 8) *reinterpret_cast<uint4 *>(drow + 256) = v1;
        }
    }
}

// bf16, F in {8, 16}, d_h % 8 == 0, 16-byte aligned: the tensor-core kernel.  Returns -100 when the shape is not eligible.
static int launch_attn_mma(const Geo &g, const bf16 *qkv, bf16 *ctx, cudaStream_t st) {
    if (!(g.F == 8 || g.F == 16) || g.dh % 8 != 0 || g.dh < 8) return -100;
    // head group: W = HB * dh as close to 320 channels as the head count allows and a multiple of 64 (bank-conflict-free rows)
    int HB = 0;
    for (int hb = g.heads; hb >= 1; hb--)
        if (g.heads % hb == 0 && (hb * g.dh) % 64 == 0 && hb * g.dh <= 320) { HB = hb; break; }
    if (HB == 0) return -100;
    // SD1.5 levels (d_h = 40 / 80 / 160, head groups of exactly 320 channels): compile-time specialised kernel
    if ((g.dh == 40 || g.dh == 80 || g.dh == 160) && HB * g.dh == 320 && (int64_t)g.F * g.P * 3 * g.C < (1ll << 31) && opt(NMM_OPT_ATTN_VARIANT) == 0) {
        const size_t row_b = (size_t)(3 * 320 + 8) * 2;
        static const int pb_env = getenv("NMM_ATTN_PB") ? atoi(getenv("NMM_ATTN_PB")) : 0;
        int PBf = pb_env > 0 ? pb_env : (int)((40 * 1024) / (g.F * row_b));
        if (PBf < 1) PBf = 1;
        if (PBf > g.P) PBf = g.P;
        if (pb_env <= 0)                                                 // small levels: more, smaller CTAs until the grid is >= 4 per SM
            while (PBf > 1 && (int64_t)g.B * ceil_div(g.P, PBf) * (g.heads / HB) < 4 * 148) PBf--;
        const size_t smem_f = (size_t)PBf * g.F * row_b;
        if (smem_f > 200 * 1024) return fail(NMM_ERR_UNSUPPORTED, "attention tile of %d positions needs %zu bytes of shared memory", PBf, smem_f);
        const int64_t nblk = (int64_t)g.B * ceil_div(g.P, PBf);
        if (nblk > 0x7fffffff) return -100;
        const dim3 gridf((unsigned)nblk, (unsigned)(g.heads / HB));
        const float sl2 = (1.0f / sqrtf((float)g.dh)) * 1.4426950408889634f;
        const int thr_f = std::min(256, std::max(128, PBf * HB * 32));      // one warp per problem, at least 4 warps for staging
#define ATTN_FIXED(FF, DD)                                                                                               \
    do {                                                                                                                 \
        auto kern = temporal_attention_mma_fixed_kernel<FF, DD>;                                                         \
        static DeviceOnce once;                                                                                          \
        NMM_CUDA_OK(once.max_smem(kern, 200 * 1024));          \
        ProfScope prof(K_ATTENTION, st, 4.0 * g.N * g.F * g.C, 4.0 * g.N * g.C * 2);                                      \
        launch_pdl(kern, gridf, thr_f, smem_f, st, qkv, ctx, g.P, g.C, PBf, sl2);                                          \
    } while (0)
        if (g.F == 8) {
            if (g.dh == 40) ATTN_FIXED(8, 40); else if (g.dh == 80) ATTN_FIXED(8, 80); else ATTN_FIXED(8, 160);
        } else {
            if (g.dh == 40) ATTN_FIXED(16, 40); else if (g.dh == 80) ATTN_FIXED(16, 80); else ATTN_FIXED(16, 160);
        }
#undef ATTN_FIXED
        NMM_LAUNCHED("temporal_attention_mma_fixed_kernel");
        return NMM_OK;
    }
    const int W = HB * g.dh;
    const size_t row_bytes = (size_t)(3 * W + 8) * 2;
    int PB = (int)((40 * 1024) / (g.F * row_bytes));                  // <= 40 KB per CTA: ~5 CTAs per SM
    if (PB < 1) PB = 1;
    if (PB > g.P) PB = g.P;
    const size_t smem = (size_t)PB * g.F * row_bytes;
    if (smem > 200 * 1024) return -100;
    int warps = PB * HB;                                               // one problem per warp per pass, at most 8 warps
    if (warps > 8) warps = 8;
    const int64_t blocks = (int64_t)g.B * ceil_div(g.P, PB);
    if (blocks > 0x7fffffff) return -100;
    const dim3 grid((unsigned)blocks, (unsigned)(g.heads / HB));
    const float scale_log2e = (1.0f / sqrtf((float)g.dh)) * 1.4426950408889634f;
#define ATTN_MMA(FF)                                                                                                     \
    do {                                                                                                                 \
        auto kern = temporal_attention_mma_kernel<FF>;                                                                   \
        static DeviceOnce once;                                                                                          \
        NMM_CUDA_OK(once.max_smem(kern, 200 * 1024));          \
        ProfScope prof(K_ATTENTION, st, 4.0 * g.N * g.F * g.C, 4.0 * g.N * g.C * 2);                                      \
        launch_pdl(kern, grid, warps * 32, smem, st, qkv, ctx, g.B, g.P, g.C, g.heads, PB, HB, scale_log2e);                      \
    } while (0)
    if (g.F == 8) ATTN_MMA(8);
    else ATTN_MMA(16);
#undef ATTN_MMA
    NMM_LAUNCHED("temporal_attention_mma_kernel");
    return NMM_OK;
}

int launch_temporal_attention(const Geo &g, const void *qkv, void *ctx, cudaStream_t st) {
    if (g.F > NMM_MAX_FRAMES) return fail(NMM_ERR_UNSUPPORTED, "frames %d > %d", g.F, NMM_MAX_FRAMES);
    const bool al = aligned(qkv, 16) && aligned(ctx, 16);
    if (g.dtype == NMM_BF16) {
        if (al && opt(NMM_OPT_ATTN_VARIANT) != 2) {
            const int rc = launch_attn_mma(g, (const bf16 *)qkv, (bf16 *)ctx, st);
            if (rc != -100) return rc;
        }
        if (g.dh % 8 == 0 && al) return launch_attn_t<bf16, 8>(g, (const bf16 *)qkv, (bf16 *)ctx, st);
        return launch_attn_t<bf16, 1>(g, (const bf16 *)qkv, (bf16 *)ctx, st);
    }
    const int split = planes_of(g.dtype) > 1 ? planes_of(g.dtype) : 0;      // the context feeds to_out's tensor-core GEMM: 2 / 3 bf16 planes
    if (g.dh % 4 == 0 && al && g.C % 4 == 0) return launch_attn_t<float, 4>(g, (const float *)qkv, (float *)ctx, st, split);
    return launch_attn_t<float, 1>(g, (const float *)qkv, (float *)ctx, st, split);
}

}  // namespace nmm

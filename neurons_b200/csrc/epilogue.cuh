// Fused GEMM epilogues shared by the fp32 FMA GEMM and the tcgen05 GEMM.
// Each call handles NC consecutive output columns of ONE row held in registers (fp32 accumulators).
//   STORE     out = acc + bias                                         Linear            motion_module.py:145, :289-298
//   RESIDUAL  h   = acc + bias + h   (or out = acc + bias + h)         "attn(...) + hidden_states", "ff(...) + hidden_states"  :213-219
//   GEGLU     out = (acc_v + b_v) * gelu_erf(acc_g + b_g)              GEGLU.forward     motion_module_new.py:516-518
//             (columns in groups of four: value 2q, value 2q+1, gate 2q, gate 2q+1 -> outputs 2q, 2q+1)
//   OUTPUT    y[b,c,f,p] = acc + bias + x[b,c,f,p]                     proj_out, back to NCHW, + residual      motion_module.py:152-156
#pragma once
#include "common.cuh"

namespace nmm {

struct EpiParams {
    int64_t M;
    int N;
    const float *bias;
    float *h;
    void *out;
    const void *x;
    void *y;
    int F, P;
    int64_t xsb, xsc, xsf, ysb, ysc, ysf;
    float2 *y_part;    // OUTPUT, nchw_vec path only: statistics of y for the next GroupNorm (LinearArgs::y_part)
    int nchw_vec;      // OUTPUT: P % 32 == 0 and x / y rows 16-byte aligned -> 8-position (16-byte) vector path
    int no_h_store;
    float *ln_part_out;
    const float *ln_part_in;
    int ln_nparts, ln_K;
    const float *ln_g, *ln_c, *ln_pew;
    float ln_eps;
};

// OUTPUT epilogue: can the bf16 16-byte vector path run (and with it the y-statistics emission)?
inline bool output_vec_ok(const LinearArgs &a) {
    return a.epilogue == NMM_EPI_OUTPUT && a.planes <= 1 && a.P > 0 && a.P % 32 == 0 && aligned(a.x, 16) && aligned(a.y, 16) && a.xsb % 8 == 0 &&
           a.xsc % 8 == 0 && a.xsf % 8 == 0 && a.ysb % 8 == 0 && a.ysc % 8 == 0 && a.ysf % 8 == 0;
}

inline EpiParams epi_params_of(const LinearArgs &a) {
    EpiParams e;
    e.M = a.M; e.N = a.N; e.bias = a.bias; e.h = a.h; e.out = a.out; e.x = a.x; e.y = a.y; e.F = a.F; e.P = a.P;
    e.xsb = a.xsb; e.xsc = a.xsc; e.xsf = a.xsf; e.ysb = a.ysb; e.ysc = a.ysc; e.ysf = a.ysf;
    e.no_h_store = a.no_h_store;
    e.y_part = a.y_part;
    e.ln_part_out = a.ln_part_out; e.ln_part_in = a.ln_part_in; e.ln_nparts = a.ln_nparts; e.ln_K = a.K;
    e.ln_g = a.ln_g; e.ln_c = a.ln_c; e.ln_pew = a.ln_pew; e.ln_eps = a.ln_eps;
    e.nchw_vec = output_vec_ok(a) ? 1 : 0;
    if (!e.nchw_vec) e.y_part = nullptr;
    return e;
}

template <int NC> __device__ __forceinline__ void store_row(float *dst, const float (&v)[NC]) {
    static_assert(NC % 4 == 0, "NC");
#pragma unroll
    for (int i = 0; i < NC / 4; i++) reinterpret_cast<float4 *>(dst)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
template <int NC> __device__ __forceinline__ void store_row(bf16 *dst, const float (&v)[NC]) {
    static_assert(NC % 4 == 0, "NC");
    if constexpr (NC % 8 == 0) {
#pragma unroll
        for (int i = 0; i < NC / 8; i++)
            reinterpret_cast<uint4 *>(dst)[i] = make_uint4(pack_bf16x2(v[8 * i], v[8 * i + 1]), pack_bf16x2(v[8 * i + 2], v[8 * i + 3]),
                                                           pack_bf16x2(v[8 * i + 4], v[8 * i + 5]), pack_bf16x2(v[8 * i + 6], v[8 * i + 7]));
    } else {
#pragma unroll
        for (int i = 0; i < NC / 4; i++)
            reinterpret_cast<uint2 *>(dst)[i] = make_uint2(pack_bf16x2(v[4 * i], v[4 * i + 1]), pack_bf16x2(v[4 * i + 2], v[4 * i + 3]));
    }
}

template <int NC> __device__ __forceinline__ void add_bias(float (&v)[NC], const float *bias, int col0) {
    if (bias == nullptr) return;
#pragma unroll
    for (int i = 0; i < NC / 4; i++) {
        float4 b = __ldg(reinterpret_cast<const float4 *>(bias + col0) + i);
        v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
    }
}

// T = element type of out / x / y (float or bf16).  Caller guarantees row < M and col0 + NC <= N.
template <int EPI, typename T, int NC>
__device__ __forceinline__ void epilogue_apply(const EpiParams &e, int64_t row, int col0, float (&acc)[NC]) {
    add_bias<NC>(acc, e.bias, col0);
    if constexpr (EPI == NMM_EPI_STORE) {
        // either / both destinations: fp32 residual stream `h`, GEMM-dtype `out`
        if (e.h != nullptr) store_row<NC>(e.h + row * e.N + col0, acc);
        if (e.out != nullptr) store_row<NC>(reinterpret_cast<T *>(e.out) + row * e.N + col0, acc);
    } else if constexpr (EPI == NMM_EPI_RESIDUAL) {
        float *hp = e.h + row * e.N + col0;
#pragma unroll
        for (int i = 0; i < NC / 4; i++) {
            float4 r = reinterpret_cast<const float4 *>(hp)[i];
            acc[4 * i] += r.x; acc[4 * i + 1] += r.y; acc[4 * i + 2] += r.z; acc[4 * i + 3] += r.w;
        }
        if (e.out != nullptr) store_row<NC>(reinterpret_cast<T *>(e.out) + row * e.N + col0, acc);
        if (!e.no_h_store) store_row<NC>(hp, acc);
    } else if constexpr (EPI == NMM_EPI_GEGLU) {
        float o[NC / 2];
#pragma unroll
        for (int q = 0; q < NC / 4; q++) {      // columns 4q .. 4q+3 = value 2q, value 2q+1, gate 2q, gate 2q+1
            o[2 * q] = acc[4 * q] * gelu_erf(acc[4 * q + 2]);
            o[2 * q + 1] = acc[4 * q + 1] * gelu_erf(acc[4 * q + 3]);
        }
        T *dst = reinterpret_cast<T *>(e.out) + row * (e.N / 2) + col0 / 2;
        if constexpr (NC / 2 >= 4) {
            store_row<NC / 2>(dst, o);
        } else {
#pragma unroll
            for (int j = 0; j < NC / 2; j++) dst[j] = from_f32<T>(o[j]);
        }
    } else {   // NMM_EPI_OUTPUT
        const int64_t bf = row / e.P;
        const int p = (int)(row - bf * e.P);
        const int64_t b = bf / e.F, f = bf - b * e.F;
        const T *xp = reinterpret_cast<const T *>(e.x) + b * e.xsb + f * e.xsf + p;
        T *yp = reinterpret_cast<T *>(e.y) + b * e.ysb + f * e.ysf + p;
#pragma unroll
        for (int j = 0; j < NC; j++) {
            const int64_t c = col0 + j;
            yp[c * e.ysc] = from_f32<T>(acc[j] + to_f32(xp[c * e.xsc]));
        }
    }
}

}  // namespace nmm

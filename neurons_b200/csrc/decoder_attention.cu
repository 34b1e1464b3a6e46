// Temporal attention of the blurry-video decoder (SURVEY 8(f) N4): the `temp_attn` + blend step of AttnUpDecoderBlock2D / UNetMidBlock2D,
// /root/reference/model_variants/video_decoder.py:237-248 and :394-406:
//     res = rearrange(x.reshape(b, t, c, h, w), 'b t c h w -> (b h w) t c')
//     res = temp_attn(res)                      # diffusers Attention(c, heads = c / head_dim, norm_num_groups = 32, residual_connection = True,
//                                               #                     bias = True, rescale_output_factor = r, _from_deprecated_attn_block = True)
//     res = rearrange(res.reshape(b, h, w, t, c), 'b h w t c -> (b t) c h w')
//     y = weight * x + (1 - weight) * res
// The Attention class is diffusers' (>= 0.20, `diffusers.models.attention_processor`; imported at video_decoder.py:2, NOT vendored and not
// installable here): its published arithmetic for a 3-D input with AttnProcessor2_0 is restated in oracle/decoder_oracle.py --
//     n = GroupNorm(32, c, eps)(res^T)^T          (statistics per sequence = per position, over the c / 32 channels of a group x the t frames)
//     q, k, v = n Wq^T + bq, n Wk^T + bk, n Wv^T + bv;   o = softmax(q k^T / sqrt(d_h)) v  per head over the t frames
//     out = (o Wo^T + bo + res) / r
// PARITY UNPINNED: no reference fixture can be generated for this block (see DESIGN.md section 8).
//
// Token order is the motion module's: x [(b t), c, h, w] IS a [B, F = t, C, H, W]-storage view, tokens n = (b * t + f) * P + p, attention per
// (b, p, head) over f -- so the block runs on the motion module's kernels: one new kernel (GroupNorm over (group channels x frames) per
// position, fused with the re-layout to tokens), the GEMM with bias for q | k | v, the temporal attention kernel (any t <= 32), and the
// OUTPUT epilogue, which writes  y = acc + b' + x  straight back in NCHW.  With r = 1 (every block of DecoderVideo) the blend folds into
// the output projection:  y = x + (1 - weight) * (o Wo^T + bo)  ->  Wo' = (1 - weight) Wo, bo' = (1 - weight) bo  at pack time.
#include <algorithm>

#include "common.cuh"

namespace nmm {
namespace {

// one thread per (b, p, group): reads its group's cpg x T values (stride P between channels, sf between frames), writes the normalised,
// affine-transformed values as token rows.  The tensors of this decoder are small (c <= 128, <= 112 x 112 positions): simplicity over peak.
template <typename T>
__global__ void __launch_bounds__(128) gn_time_tokens_kernel(const T *__restrict__ x, const float *__restrict__ gamma, const float *__restrict__ beta,
                                                            T *__restrict__ tokens, int B, int C, int F, int P, float eps, int64_t sb, int64_t sc,
                                                            int64_t sf) {
    pdl_wait();
    pdl_launch_dependents();
    const int cpg = C / NMM_GN_GROUPS;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;          // ((b * 32 + g) * P + p): consecutive threads = consecutive positions
    if (i >= (int64_t)B * NMM_GN_GROUPS * P) return;
    const int p = (int)(i % P), g = (int)((i / P) % NMM_GN_GROUPS), b = (int)(i / ((int64_t)P * NMM_GN_GROUPS));
    const T *xb = x + (int64_t)b * sb + p;
    // The frames of a decoded video are close to each other, so a group (cpg channels x t frames at one position) often has a variance
    // far below mean^2, where sq / n - mean^2 on raw values cancels away every significant bit.  Shifting by the group's first value K
    // keeps the sums of v - K well conditioned, and the values are normalised as (v - K) - mean_d without rounding the mean K + mean_d.
    const float K = to_f32(xb[(int64_t)(g * cpg) * sc]);
    float sum = 0.f, sq = 0.f;
    for (int f = 0; f < F; f++)
        for (int j = 0; j < cpg; j++) {
            const float d = to_f32(xb[(int64_t)f * sf + (int64_t)(g * cpg + j) * sc]) - K;
            sum += d; sq = fmaf(d, d, sq);
        }
    const float n = (float)(F * cpg);
    const float mean_d = sum / n;
    const float var = fmaxf(sq / n - mean_d * mean_d, 0.f);
    const float rstd = rsqrtf(var + eps);
    for (int f = 0; f < F; f++)
        for (int j = 0; j < cpg; j++) {
            const int c = g * cpg + j;
            const float d = to_f32(xb[(int64_t)f * sf + (int64_t)c * sc]) - K;
            tokens[((int64_t)(b * F + f) * P + p) * C + c] = from_f32<T>((d - mean_d) * rstd * gamma[c] + beta[c]);
        }
}

// dst = scale * src (fp32 -> fp32 or bf16): the blend factor folded into the output projection
template <typename TS, typename TD>
__global__ void scale_convert_kernel(const TS *__restrict__ src, TD *__restrict__ dst, int64_t n, float scale) {
    pdl_wait();
    pdl_launch_dependents();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = from_f32<TD>(scale * to_f32(src[i]));
}
int scale_convert(const void *src, int sd, void *dst, int dd, int64_t n, float scale, cudaStream_t st) {
    if (!src || !dst) return fail(NMM_ERR_BAD_ARG, "NULL parameter tensor");
    const int blocks = (int)std::min<int64_t>(ceil_div(n, 256), 148 * 8);
    if (sd == NMM_F32 && dd == NMM_F32) launch_pdl(scale_convert_kernel<float, float>, blocks, 256, 0, st, (const float *)src, (float *)dst, n, scale);
    else if (sd == NMM_F32 && dd == NMM_BF16) launch_pdl(scale_convert_kernel<float, bf16>, blocks, 256, 0, st, (const float *)src, (bf16 *)dst, n, scale);
    else if (sd == NMM_BF16 && dd == NMM_F32) launch_pdl(scale_convert_kernel<bf16, float>, blocks, 256, 0, st, (const bf16 *)src, (float *)dst, n, scale);
    else if (sd == NMM_BF16 && dd == NMM_BF16) launch_pdl(scale_convert_kernel<bf16, bf16>, blocks, 256, 0, st, (const bf16 *)src, (bf16 *)dst, n, scale);
    else return fail(NMM_ERR_BAD_ARG, "unknown parameter dtype");
    NMM_LAUNCHED("scale_convert_kernel");
    return NMM_OK;
}

struct DaLayout { size_t gn_w, gn_b, wqkv, bqkv, wo, bo, total; };
DaLayout da_layout(int C, int dtype) {
    DaLayout L;
    size_t off = 0;
    const size_t c = C, ws = dtype_size(dtype);
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    L.gn_w = take(c * 4); L.gn_b = take(c * 4);
    L.wqkv = take(3 * c * c * ws); L.bqkv = take(3 * c * 4);
    L.wo = take(c * c * ws); L.bo = take(c * 4);
    L.total = off;
    return L;
}
struct DaWork { size_t tok, qkv, ctx, total; };
DaWork da_work(const Geo &g) {
    DaWork w;
    size_t off = 0;
    const size_t es = dtype_size(g.dtype), N = (size_t)g.N, C = g.C;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
    w.tok = take(N * C * es); w.qkv = take(N * 3 * C * es); w.ctx = take(N * C * std::max<size_t>(es, 4));
    w.total = off;
    return w;
}
int da_validate(const nmm_shape *s, nmm_shape *norm) {
    if (!s) return fail(NMM_ERR_BAD_ARG, "shape is NULL");
    *norm = *s;
    norm->layers = 1; norm->attn_blocks = 1; norm->pos_enc = 0; norm->max_len = 0; norm->ln_fold = 0;
    int rc = nmm_validate(norm);
    if (rc != NMM_OK) return rc;
    if (s->dtype != NMM_F32 && s->dtype != NMM_BF16) return fail(NMM_ERR_UNSUPPORTED, "decoder temporal attention: dtype must be NMM_F32 or NMM_BF16");
    if (s->dtype == NMM_BF16 && s->channels % 32 != 0) return fail(NMM_ERR_UNSUPPORTED, "bf16 mode needs channels %% 32 == 0");
    return NMM_OK;
}

}  // namespace
}  // namespace nmm

using namespace nmm;

extern "C" {

int nmm_decoder_attn_packed_bytes(int32_t channels, int32_t dtype, size_t *out_bytes) {
    if (channels <= 0 || !out_bytes || (dtype != NMM_F32 && dtype != NMM_BF16)) return fail(NMM_ERR_BAD_ARG, "bad argument");
    *out_bytes = da_layout(channels, dtype).total;
    return NMM_OK;
}

int nmm_decoder_attn_workspace_bytes(const nmm_shape *s, size_t *out_bytes) {
    nmm_shape n;
    int rc = da_validate(s, &n);
    if (rc != NMM_OK) return rc;
    if (!out_bytes) return fail(NMM_ERR_BAD_ARG, "out_bytes is NULL");
    *out_bytes = da_work(geo_of(&n)).total;
    return NMM_OK;
}

int nmm_decoder_attn_pack(int32_t channels, int32_t dtype, const nmm_decoder_attn_params *src, float blend_weight, float rescale_output_factor,
                          void *packed, size_t packed_bytes, void *stream) {
    if (channels <= 0 || !src || !packed || (dtype != NMM_F32 && dtype != NMM_BF16)) return fail(NMM_ERR_BAD_ARG, "bad argument");
    if (src->dtype != NMM_F32 && src->dtype != NMM_BF16) return fail(NMM_ERR_BAD_ARG, "unknown source parameter dtype %d", src->dtype);
    if (rescale_output_factor != 1.0f)
        return fail(NMM_ERR_UNSUPPORTED, "decoder temporal attention: rescale_output_factor %g != 1 (every block of the reference's DecoderVideo uses 1)",
                    rescale_output_factor);
    int rc = device_check();
    if (rc != NMM_OK) return rc;
    const DaLayout L = da_layout(channels, dtype);
    if (packed_bytes < L.total) return fail(NMM_ERR_WORKSPACE, "packed buffer too small: %zu < %zu", packed_bytes, L.total);
    if (!aligned(packed, 256)) return fail(NMM_ERR_BAD_ARG, "packed buffer must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char *base = (char *)packed;
    const int sd = src->dtype;
    const int64_t C = channels;
    const size_t ws = dtype_size(dtype);
#define PACK(srcp, off, dd, rows, cols)                                                              \
    do {                                                                                             \
        rc = launch_convert_rows((srcp), sd, base + (off), (dd), (rows), (cols), 0, st);             \
        if (rc != NMM_OK) return rc;                                                                 \
    } while (0)
    PACK(src->gn_w, L.gn_w, NMM_F32, C, 1); PACK(src->gn_b, L.gn_b, NMM_F32, C, 1);
    PACK(src->to_q_w, L.wqkv, dtype, C, C); PACK(src->to_k_w, L.wqkv + (size_t)C * C * ws, dtype, C, C); PACK(src->to_v_w, L.wqkv + 2 * (size_t)C * C * ws, dtype, C, C);
    PACK(src->to_q_b, L.bqkv, NMM_F32, C, 1); PACK(src->to_k_b, L.bqkv + (size_t)C * 4, NMM_F32, C, 1); PACK(src->to_v_b, L.bqkv + 2 * (size_t)C * 4, NMM_F32, C, 1);
#undef PACK
    // y = weight * x + (1 - weight) * (o Wo^T + bo + x) = x + (1 - weight) * (o Wo^T + bo)      (video_decoder.py:248 with r = 1)
    const float s = 1.0f - blend_weight;
    if ((rc = scale_convert(src->to_out_w, sd, base + L.wo, dtype, C * C, s, st)) != NMM_OK) return rc;
    return scale_convert(src->to_out_b, sd, base + L.bo, NMM_F32, C, s, st);
}

int nmm_decoder_temporal_attention(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace,
                                   size_t workspace_bytes, void *stream) {
    nmm_shape n;
    int rc = da_validate(s, &n);
    if (rc != NMM_OK) return rc;
    if (!x || !y || !packed || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if (x == y) return fail(NMM_ERR_BAD_ARG, "x and y must not alias");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(&n);
    const DaLayout L = da_layout(g.C, g.dtype);
    const DaWork w = da_work(g);
    if (packed_bytes != L.total) return fail(NMM_ERR_WORKSPACE, "packed parameter buffer of %zu bytes does not match this call's layout (%zu bytes)", packed_bytes, L.total);
    if (workspace_bytes < w.total) return fail(NMM_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, w.total);
    if (!aligned(workspace, 1024) || !aligned(packed, 256)) return fail(NMM_ERR_BAD_ARG, "workspace must be 1024-byte and packed params 256-byte aligned");
    if ((int64_t)g.B * NMM_GN_GROUPS * g.P > ((int64_t)1 << 31)) return fail(NMM_ERR_UNSUPPORTED, "tensor too large");
    cudaStream_t st = (cudaStream_t)stream;
    const char *pk = (const char *)packed;
    char *ws = (char *)workspace;
    void *tok = ws + w.tok, *qkv = ws + w.qkv, *ctx = ws + w.ctx;
    auto F32 = [&](size_t off) { return (const float *)(pk + off); };

    // GroupNorm over (group channels x frames) per position + re-layout to tokens            Attention.group_norm on [B', c, t]
    {
        const int64_t threads = (int64_t)g.B * NMM_GN_GROUPS * g.P;
        const unsigned blocks = (unsigned)ceil_div(threads, 128);
        ProfScope prof(K_GN_TOKENS, st, 0.0, 2.0 * g.N * g.C * dtype_size(g.dtype));
        if (g.dtype == NMM_BF16)
            launch_pdl(gn_time_tokens_kernel<bf16>, blocks, 128, 0, st, (const bf16 *)x, F32(L.gn_w), F32(L.gn_b), (bf16 *)tok, g.B, g.C, g.F, g.P, s->eps_gn,
                       s->x_stride_b, s->x_stride_c, s->x_stride_f);
        else
            launch_pdl(gn_time_tokens_kernel<float>, blocks, 128, 0, st, (const float *)x, F32(L.gn_w), F32(L.gn_b), (float *)tok, g.B, g.C, g.F, g.P, s->eps_gn,
                       s->x_stride_b, s->x_stride_c, s->x_stride_f);
        NMM_LAUNCHED("gn_time_tokens_kernel");
    }
    LinearArgs a;
    memset(&a, 0, sizeof(a));
    a.M = g.N; a.F = g.F; a.P = g.P;
    a.xsb = s->x_stride_b; a.xsc = s->x_stride_c; a.xsf = s->x_stride_f;
    a.ysb = s->y_stride_b; a.ysc = s->y_stride_c; a.ysf = s->y_stride_f;
    // q | k | v with bias                                                                      to_q / to_k / to_v (bias = True)
    a.epilogue = NMM_EPI_STORE; a.N = 3 * g.C; a.K = g.C; a.A = tok; a.W = pk + L.wqkv; a.bias = F32(L.bqkv); a.h = nullptr; a.out = qkv;
    if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
    // softmax(q k^T / sqrt(d_h)) v over the frames of each position                            F.scaled_dot_product_attention
    if ((rc = launch_temporal_attention(g, qkv, ctx, st)) != NMM_OK) return rc;
    // y = x + (1 - weight) * (o Wo^T + bo), back in [(b t), c, h, w]                           to_out[0] + residual, then the blend (:248)
    a.epilogue = NMM_EPI_OUTPUT; a.N = g.C; a.K = g.C; a.A = ctx; a.W = pk + L.wo; a.bias = F32(L.bo); a.out = nullptr; a.x = x; a.y = y;
    return linear_dispatch(g.dtype, a, st);
}

}  // extern "C"

// C ABI of the spatial transformer (SURVEY 8(f) N3): Transformer3DModel.forward of the UNet's CrossAttn blocks,
// /root/reference/animatediff/models/attention.py:95-148 (-> BasicTransformerBlock.forward :258-300) with the inherited
// CrossAttention / FeedForward / GEGLU arithmetic (diffusers 0.11.1; in-tree copy motion_module_new.py:119-339,429-534).
// NEURONS configuration (SD1.5 topology, unet.py:157-183): Conv2d 1x1 proj_in / proj_out (use_linear_projection = False), one
// BasicTransformerBlock per model, LayerNorm (no AdaLayerNorm), attention_bias = False, unet_use_cross_frame_attention = False,
// unet_use_temporal_attention = False, cross_attention_dim = 768, GEGLU feed-forward, no attention mask.
//
// The module has the motion module's skeleton -- GroupNorm -> proj_in -> [LN -> attention -> +h]* -> LN -> GEGLU FF -> +h -> proj_out
// -> + x -- in the SAME token order n = (b*F + f)*P + p (attention.py:100,111 "(b f) (h w) c"), so it runs on the motion module's
// kernels: gn_stats, GroupNorm (+) re-layout (+) proj_in in one tcgen05 kernel (a 1x1 convolution is the same [C, C] GEMM),
// layernorm, the tcgen05 GEMM with STORE / RESIDUAL / GEGLU / OUTPUT epilogues (proj_out writes y = acc + b + x straight into the
// [B, F, C, H, W] storage that attention.py:144 returns as a view).  What it adds is attention over the P positions of a frame
// (and over the 77 text tokens) instead of over the frames of a position: spatial_attention.cu.
#include <algorithm>

#include "common.cuh"
#include "epilogue.cuh"

namespace nmm {
namespace {

struct SpLayerOff { size_t ln1_w, ln1_b, wqkv1, wo1, bo1, ln2_w, ln2_b, wq2, wkv2, wo2, bo2, ln3_w, ln3_b, w1, b1, w2, b2; };
struct SpLayout {
    size_t header, gn_w, gn_b, w_in, b_in;
    SpLayerOff layer[NMM_MAX_LAYERS];
    size_t w_out, b_out, total;
};
struct SpHeader { uint32_t magic, abi; int32_t dtype, C, heads, layers, ctx_dim, pad; uint64_t total; uint64_t reserved[3]; };
static_assert(sizeof(SpHeader) == 64, "spatial packed header is 64 bytes");
constexpr uint32_t SP_MAGIC = 0x4D4D4E53u;      // "SNMM"

__global__ void sp_write_header_kernel(SpHeader hd, SpHeader *dst) {
    pdl_wait();
    pdl_launch_dependents();
    if (threadIdx.x == 0 && blockIdx.x == 0) *dst = hd;
}

SpLayout sp_layout(const Geo &g, int ctx_dim) {
    SpLayout L;
    memset(&L, 0, sizeof(L));
    size_t off = 0;
    const size_t C = g.C, D = ctx_dim, ws = g.dtype == NMM_F32X3 ? 4 : dtype_size(g.dtype);      // X3: bf16 [rows, 2 * cols]
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    L.header = take(sizeof(SpHeader));
    L.gn_w = take(C * 4); L.gn_b = take(C * 4);
    L.w_in = take(C * C * ws); L.b_in = take(C * 4);
    for (int l = 0; l < g.layers; l++) {
        SpLayerOff &o = L.layer[l];
        o.ln1_w = take(C * 4); o.ln1_b = take(C * 4);
        o.wqkv1 = take(3 * C * C * ws); o.wo1 = take(C * C * ws); o.bo1 = take(C * 4);
        o.ln2_w = take(C * 4); o.ln2_b = take(C * 4);
        o.wq2 = take(C * C * ws); o.wkv2 = take(2 * C * D * ws); o.wo2 = take(C * C * ws); o.bo2 = take(C * 4);
        o.ln3_w = take(C * 4); o.ln3_b = take(C * 4);
        o.w1 = take(8 * C * C * ws); o.b1 = take(8 * C * 4);
        o.w2 = take(4 * C * C * ws); o.b2 = take(C * 4);
    }
    L.w_out = take(C * C * ws); L.b_out = take(C * 4);
    L.total = off;
    return L;
}

struct SpWork { size_t gn_partial, tok, h, big, ctx, kv, stat_part, ctx32, ehs2, qkv2, kv2, total; };
SpWork sp_work(const Geo &g, int ctx_len, int ctx_dim) {
    SpWork w;
    size_t off = 0;
    const size_t es = dtype_size(g.dtype);
    const size_t opnd = g.dtype == NMM_F32X3 ? 4 : es;      // GEMM-operand element bytes (X3: two bf16 planes)
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
    const size_t N = (size_t)g.N, C = g.C;
    w.gn_partial = take(gn_partial_bytes(g));
    w.tok = take(N * C * opnd);
    w.h = take(N * C * 4);
    w.big = take(N * 4 * C * std::max(opnd, es));
    w.ctx = take(N * C * std::max(opnd, es));
    w.kv = take((size_t)g.B * ctx_len * 2 * C * 4);
    w.stat_part = take((N + 31) / 32 * C * sizeof(float2));      // N1: (sum, sum of squares) partials of y per 32-row block and channel
    // NMM_F32X3: the fp32 attention output before it is split into hi | lo planes; the text states as hi | lo planes
    w.ctx32 = take(g.dtype == NMM_F32X3 ? N * C * 4 : 0);
    w.ehs2 = take(g.dtype == NMM_F32X3 ? (size_t)g.B * ctx_len * ctx_dim * 4 : 0);
    // ... and q | k | v (self-attention) / q (cross-attention) and the text k | v as hi | lo planes for the fp32-grade attention kernel
    w.qkv2 = take(g.dtype == NMM_F32X3 ? N * 3 * C * 4 : 0);
    w.kv2 = take(g.dtype == NMM_F32X3 ? (size_t)g.B * ctx_len * 2 * C * 4 : 0);
    w.total = off;
    return w;
}

int sp_validate(const nmm_spatial_shape *s) {
    if (!s) return fail(NMM_ERR_BAD_ARG, "shape is NULL");
    nmm_shape b = s->base;
    b.attn_blocks = 1; b.pos_enc = 0; b.max_len = 0; b.ln_fold = 0;
    int rc = nmm_validate(&b);
    if (rc != NMM_OK) return rc;
    if (b.dtype == NMM_F32X3 && s->ctx_dim % 64 != 0) return fail(NMM_ERR_UNSUPPORTED, "NMM_F32X3 needs ctx_dim %% 64 == 0 (got %d); use NMM_F32", s->ctx_dim);
    if (s->ctx_len <= 0 || s->ctx_dim <= 0 || s->ctx_dim % 8 != 0) return fail(NMM_ERR_BAD_ARG, "ctx_len / ctx_dim must be positive, ctx_dim %% 8 == 0");
    const int dh = b.channels / b.heads;
    if (dh != 40 && dh != 80 && dh != 160) return fail(NMM_ERR_UNSUPPORTED, "spatial transformer: head dim %d (supported: 40, 80, 160)", dh);
    if (b.dtype == NMM_BF16 && b.channels % 32 != 0) return fail(NMM_ERR_UNSUPPORTED, "bf16 mode needs channels %% 32 == 0");
    return NMM_OK;
}

Geo sp_geo(const nmm_spatial_shape *s) {
    nmm_shape b = s->base;
    b.attn_blocks = 1; b.pos_enc = 0; b.max_len = 0; b.ln_fold = 0;
    return geo_of(&b);
}

}  // namespace
}  // namespace nmm

using namespace nmm;

extern "C" {

int nmm_spatial_packed_params_bytes(const nmm_spatial_shape *s, size_t *out_bytes) {
    int rc = sp_validate(s);
    if (rc != NMM_OK) return rc;
    if (!out_bytes) return fail(NMM_ERR_BAD_ARG, "out_bytes is NULL");
    *out_bytes = sp_layout(sp_geo(s), s->ctx_dim).total;
    return NMM_OK;
}

int nmm_spatial_workspace_bytes(const nmm_spatial_shape *s, size_t *out_bytes) {
    int rc = sp_validate(s);
    if (rc != NMM_OK) return rc;
    if (!out_bytes) return fail(NMM_ERR_BAD_ARG, "out_bytes is NULL");
    *out_bytes = sp_work(sp_geo(s), s->ctx_len, s->ctx_dim).total;
    return NMM_OK;
}

int nmm_spatial_pack_params(const nmm_spatial_shape *s, const nmm_spatial_params *src, void *packed, size_t packed_bytes, void *stream) {
    int rc = sp_validate(s);
    if (rc != NMM_OK) return rc;
    if (!src || !packed) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if (src->dtype != NMM_F32 && src->dtype != NMM_BF16) return fail(NMM_ERR_BAD_ARG, "unknown source parameter dtype %d", src->dtype);
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = sp_geo(s);
    const SpLayout L = sp_layout(g, s->ctx_dim);
    if (packed_bytes < L.total) return fail(NMM_ERR_WORKSPACE, "packed buffer too small: %zu < %zu", packed_bytes, L.total);
    if (!aligned(packed, 256)) return fail(NMM_ERR_BAD_ARG, "packed buffer must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char *base = (char *)packed;
    const int sd = src->dtype, wd = g.dtype;
    const int64_t C = g.C, D = s->ctx_dim;
#define PACK(srcp, off, dd, rows, cols, half)                                                        \
    do {                                                                                             \
        rc = launch_convert_rows((srcp), sd, base + (off), (dd), (rows), (cols), (half), st);        \
        if (rc != NMM_OK) return rc;                                                                 \
    } while (0)
    {
        SpHeader hd;
        memset(&hd, 0, sizeof(hd));
        hd.magic = SP_MAGIC; hd.abi = NMM_ABI_VERSION; hd.dtype = g.dtype; hd.C = g.C; hd.heads = g.heads; hd.layers = g.layers; hd.ctx_dim = s->ctx_dim;
        hd.total = L.total;
        launch_pdl(sp_write_header_kernel, 1, 32, 0, st, hd, (SpHeader *)(base + L.header));
        NMM_LAUNCHED("sp_write_header_kernel");
    }
    const size_t wsz = wd == NMM_F32X3 ? 4 : dtype_size(wd);      // X3: a row is its hi plane | lo plane (2 x bf16 per element)
    PACK(src->gn_w, L.gn_w, NMM_F32, C, 1, 0); PACK(src->gn_b, L.gn_b, NMM_F32, C, 1, 0);
    PACK(src->proj_in_w, L.w_in, wd, C, C, 0); PACK(src->proj_in_b, L.b_in, NMM_F32, C, 1, 0);      // Conv2d [C, C, 1, 1] == Linear [C, C]
    for (int l = 0; l < g.layers; l++) {
        const nmm_spatial_layer_params &lp = src->layer[l];
        const SpLayerOff &o = L.layer[l];
        PACK(lp.norm1_w, o.ln1_w, NMM_F32, C, 1, 0); PACK(lp.norm1_b, o.ln1_b, NMM_F32, C, 1, 0);
        PACK(lp.attn1_q, o.wqkv1, wd, C, C, 0); PACK(lp.attn1_k, o.wqkv1 + (size_t)C * C * wsz, wd, C, C, 0); PACK(lp.attn1_v, o.wqkv1 + 2 * (size_t)C * C * wsz, wd, C, C, 0);
        PACK(lp.attn1_out_w, o.wo1, wd, C, C, 0); PACK(lp.attn1_out_b, o.bo1, NMM_F32, C, 1, 0);
        PACK(lp.norm2_w, o.ln2_w, NMM_F32, C, 1, 0); PACK(lp.norm2_b, o.ln2_b, NMM_F32, C, 1, 0);
        PACK(lp.attn2_q, o.wq2, wd, C, C, 0);
        PACK(lp.attn2_k, o.wkv2, wd, C, D, 0); PACK(lp.attn2_v, o.wkv2 + (size_t)C * D * wsz, wd, C, D, 0);
        PACK(lp.attn2_out_w, o.wo2, wd, C, C, 0); PACK(lp.attn2_out_b, o.bo2, NMM_F32, C, 1, 0);
        PACK(lp.norm3_w, o.ln3_w, NMM_F32, C, 1, 0); PACK(lp.norm3_b, o.ln3_b, NMM_F32, C, 1, 0);
        PACK(lp.ff_proj_w, o.w1, wd, 8 * C, C, (int)(4 * C)); PACK(lp.ff_proj_b, o.b1, NMM_F32, 8 * C, 1, (int)(4 * C));
        PACK(lp.ff_out_w, o.w2, wd, C, 4 * C, 0); PACK(lp.ff_out_b, o.b2, NMM_F32, C, 1, 0);
    }
    PACK(src->proj_out_w, L.w_out, wd, C, C, 0); PACK(src->proj_out_b, L.b_out, NMM_F32, C, 1, 0);
#undef PACK
    return NMM_OK;
}

int nmm_spatial_attention(int32_t dtype, const void *q, const void *k, const void *v, void *o, int64_t q_row_stride, int64_t kv_row_stride,
                          int64_t o_row_stride, int64_t q_image_stride, int64_t kv_image_stride, int64_t o_image_stride, int32_t q_len,
                          int32_t kv_len, int32_t heads, int32_t head_dim, int32_t images, int32_t kv_div, void *stream) {
    int rc = device_check();
    if (rc != NMM_OK) return rc;
    if (!q || !k || !v || !o) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if (head_dim <= 0) return fail(NMM_ERR_BAD_ARG, "head_dim must be positive");
    FlashArgs a;
    memset(&a, 0, sizeof(a));
    a.q = q; a.k = k; a.v = v; a.o = o;
    a.q_rs = q_row_stride; a.kv_rs = kv_row_stride; a.o_rs = o_row_stride; a.q_bs = q_image_stride; a.kv_bs = kv_image_stride; a.o_bs = o_image_stride;
    a.Lq = q_len; a.Lkv = kv_len; a.heads = heads; a.images = images; a.kv_div = kv_div; a.dh = head_dim; a.dtype = dtype;
    a.scale = 1.0f / sqrtf((float)head_dim);
    a.scale_log2e = a.scale * 1.4426950408889634f;
    if (dtype == NMM_F32X3) {      // q, k, v: bf16 hi | lo planes, the lo plane half a row stride after the hi plane (spatial_forward_impl's layout); o: fp32
        if (q_row_stride % 2 || kv_row_stride % 2) return fail(NMM_ERR_BAD_ARG, "NMM_F32X3 spatial attention: row strides must be even (hi | lo planes)");
        a.q_lo_off = q_row_stride / 2; a.kv_lo_off = kv_row_stride / 2;
        return launch_spatial_attention_x3(a, (cudaStream_t)stream);
    }
    return launch_spatial_attention(a, (cudaStream_t)stream);
}

static int spatial_forward_impl(const nmm_spatial_shape *s, const void *x, const void *encoder_hidden_states, void *y, const void *packed, size_t packed_bytes,
                                void *workspace, size_t workspace_bytes, double *y_sums, void *stream) {
    int rc = sp_validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !y || !packed || !workspace || !encoder_hidden_states) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if (x == y) return fail(NMM_ERR_BAD_ARG, "x and y must not alias");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = sp_geo(s);
    const nmm_shape *bs = &s->base;
    const SpLayout L = sp_layout(g, s->ctx_dim);
    const SpWork w = sp_work(g, s->ctx_len, s->ctx_dim);
    if (packed_bytes != L.total)
        return fail(NMM_ERR_WORKSPACE, "packed parameter buffer of %zu bytes does not match this call's layout (%zu bytes): packed for another dtype / geometry?",
                    packed_bytes, L.total);
    if (workspace_bytes < w.total) return fail(NMM_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, w.total);
    if (!aligned(workspace, 1024) || !aligned(packed, 256)) return fail(NMM_ERR_BAD_ARG, "workspace must be 1024-byte and packed params 256-byte aligned");
    if (g.dtype == NMM_BF16 && !aligned(encoder_hidden_states, 16)) return fail(NMM_ERR_BAD_ARG, "encoder_hidden_states must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const char *pk = (const char *)packed;
    char *ws = (char *)workspace;
    double *gn_partial = (double *)(ws + w.gn_partial);
    void *tok = ws + w.tok, *big = ws + w.big, *ctx = ws + w.ctx, *kv = ws + w.kv;
    float *h = (float *)(ws + w.h);
    auto F32 = [&](size_t off) { return (const float *)(pk + off); };
    const int C = g.C, D = s->ctx_dim, Lc = s->ctx_len, P = g.P;
    const int64_t N = g.N;
    const size_t es = dtype_size(g.dtype);

    // GroupNorm(32, C, eps 1e-6) per (b, f) image                                        attention.py:106
    if ((rc = launch_gn_stats(g, bs, x, gn_partial, st)) != NMM_OK) return rc;
    const bool gn_fused = g.dtype == NMM_BF16 && linear_tc_gn_fusable(N, P, x, bs->x_stride_b, bs->x_stride_c, bs->x_stride_f);
    if (!gn_fused && (rc = launch_gn_tokens(g, bs, g, x, gn_partial, F32(L.gn_w), F32(L.gn_b), tok, st, 0)) != NMM_OK) return rc;

    LinearArgs a;
    memset(&a, 0, sizeof(a));
    a.M = N; a.F = g.F; a.P = P;
    a.xsb = bs->x_stride_b; a.xsc = bs->x_stride_c; a.xsf = bs->x_stride_f;
    a.ysb = bs->y_stride_b; a.ysc = bs->y_stride_c; a.ysf = bs->y_stride_f;
    // proj_in (1x1 convolution == per-token Linear) -> fp32 residual stream h            :107-110
    a.epilogue = NMM_EPI_STORE; a.N = C; a.K = C; a.A = tok; a.W = pk + L.w_in; a.bias = F32(L.b_in); a.h = h; a.out = nullptr;
    if (gn_fused) {
        a.A = nullptr; a.gn_x = x; a.gn_partial = gn_partial; a.gn_splits = gn_splits_of(g);
        a.gn_count = (double)(C / NMM_GN_GROUPS) * P; a.gn_eps = bs->eps_gn; a.gn_w = F32(L.gn_w); a.gn_b = F32(L.gn_b); a.gn_B = g.B;
    }
    if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
    a.gn_x = nullptr;

    // NMM_F32X3 (fp32 activations, every Linear on the tensor cores as 3 bf16 MMAs): GEMM operands are hi | lo bf16 planes; q, k, v come out of
    // their GEMMs as plain fp32 (STORE -> h-type buffer), the fp32 attention kernel's output is split into planes for to_out
    const bool x3 = g.dtype == NMM_F32X3;
    float *ctx32 = (float *)(ws + w.ctx32);
    const void *ehs_op = encoder_hidden_states;
    if (x3) {
        if ((rc = launch_convert_rows(encoder_hidden_states, NMM_F32, ws + w.ehs2, NMM_F32X3, (int64_t)g.B * Lc, D, 0, st)) != NMM_OK) return rc;
        ehs_op = ws + w.ehs2;
    }
    FlashArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.heads = g.heads; fa.dh = g.dh; fa.dtype = x3 ? NMM_F32 : g.dtype; fa.images = g.B * g.F; fa.Lq = P;
    fa.scale = 1.0f / sqrtf((float)g.dh); fa.scale_log2e = fa.scale * 1.4426950408889634f;

    for (int l = 0; l < g.layers; l++) {
        const SpLayerOff &o = L.layer[l];
        // ---- attn1: self-attention over the P positions of each frame                  :262-280
        if ((rc = launch_layernorm_pe(g, bs, h, F32(o.ln1_w), F32(o.ln1_b), nullptr, tok, st)) != NMM_OK) return rc;
        a.epilogue = NMM_EPI_STORE; a.M = N; a.N = 3 * C; a.K = C; a.A = tok; a.W = pk + o.wqkv1; a.bias = nullptr; a.h = nullptr; a.out = big;
        if (x3) { a.h = (float *)big; a.out = nullptr; }
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
        fa.q = big; fa.k = (const char *)big + (size_t)C * es; fa.v = (const char *)big + 2 * (size_t)C * es; fa.o = x3 ? (void *)ctx32 : ctx;
        fa.q_rs = fa.kv_rs = 3 * C; fa.o_rs = C; fa.q_bs = fa.kv_bs = (int64_t)P * 3 * C; fa.o_bs = (int64_t)P * C;
        fa.Lkv = P; fa.kv_div = 1;
        if (x3) {          // q | k | v fp32 [N, 3C] -> planes [N, 6C] (hi: q | k | v, lo: q | k | v), fp32-grade attention on the tensor cores
            bf16 *qkv2 = (bf16 *)(ws + w.qkv2);
            if ((rc = launch_convert_rows(big, NMM_F32, qkv2, NMM_F32X3, N, 3 * C, 0, st)) != NMM_OK) return rc;
            fa.q = qkv2; fa.k = qkv2 + C; fa.v = qkv2 + 2 * C;
            fa.q_rs = fa.kv_rs = 6 * C; fa.q_bs = fa.kv_bs = (int64_t)P * 6 * C; fa.q_lo_off = fa.kv_lo_off = 3 * C;
            if ((rc = launch_spatial_attention_x3(fa, st)) != NMM_OK) return rc;
        } else if ((rc = launch_spatial_attention(fa, st)) != NMM_OK) return rc;
        if (x3 && (rc = launch_convert_rows(ctx32, NMM_F32, ctx, NMM_F32X3, N, C, 0, st)) != NMM_OK) return rc;
        a.epilogue = NMM_EPI_RESIDUAL; a.N = C; a.K = C; a.A = ctx; a.W = pk + o.wo1; a.bias = F32(o.bo1); a.h = h; a.out = nullptr;
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;

        // ---- attn2: cross-attention onto the text tokens (k, v once per clip)          :282-292
        a.epilogue = NMM_EPI_STORE; a.M = (int64_t)g.B * Lc; a.N = 2 * C; a.K = D; a.A = ehs_op; a.W = pk + o.wkv2; a.bias = nullptr;
        a.h = nullptr; a.out = kv;
        if (x3) { a.h = (float *)kv; a.out = nullptr; }
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
        if ((rc = launch_layernorm_pe(g, bs, h, F32(o.ln2_w), F32(o.ln2_b), nullptr, tok, st)) != NMM_OK) return rc;
        a.epilogue = NMM_EPI_STORE; a.M = N; a.N = C; a.K = C; a.A = tok; a.W = pk + o.wq2; a.bias = nullptr; a.h = nullptr; a.out = big;
        if (x3) { a.h = (float *)big; a.out = nullptr; }
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
        fa.q = big; fa.k = kv; fa.v = (const char *)kv + (size_t)C * es; fa.o = x3 ? (void *)ctx32 : ctx;
        fa.q_rs = C; fa.kv_rs = 2 * C; fa.o_rs = C; fa.q_bs = (int64_t)P * C; fa.kv_bs = (int64_t)Lc * 2 * C; fa.o_bs = (int64_t)P * C;
        fa.Lkv = Lc; fa.kv_div = g.F;
        if (x3) {
            bf16 *q2 = (bf16 *)(ws + w.qkv2), *kv2 = (bf16 *)(ws + w.kv2);
            if ((rc = launch_convert_rows(big, NMM_F32, q2, NMM_F32X3, N, C, 0, st)) != NMM_OK) return rc;
            if ((rc = launch_convert_rows(kv, NMM_F32, kv2, NMM_F32X3, (int64_t)g.B * Lc, 2 * C, 0, st)) != NMM_OK) return rc;
            fa.q = q2; fa.k = kv2; fa.v = kv2 + C;
            fa.q_rs = 2 * C; fa.q_bs = (int64_t)P * 2 * C; fa.q_lo_off = C;
            fa.kv_rs = 4 * C; fa.kv_bs = (int64_t)Lc * 4 * C; fa.kv_lo_off = 2 * C;
            if ((rc = launch_spatial_attention_x3(fa, st)) != NMM_OK) return rc;
        } else if ((rc = launch_spatial_attention(fa, st)) != NMM_OK) return rc;
        if (x3 && (rc = launch_convert_rows(ctx32, NMM_F32, ctx, NMM_F32X3, N, C, 0, st)) != NMM_OK) return rc;
        a.epilogue = NMM_EPI_RESIDUAL; a.N = C; a.K = C; a.A = ctx; a.W = pk + o.wo2; a.bias = F32(o.bo2); a.h = h; a.out = nullptr;
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;

        // ---- feed-forward: LayerNorm -> GEGLU -> Linear, + h                            :295; motion_module_new.py:441-471,497-518
        if ((rc = launch_layernorm_pe(g, bs, h, F32(o.ln3_w), F32(o.ln3_b), nullptr, tok, st)) != NMM_OK) return rc;
        a.epilogue = NMM_EPI_GEGLU; a.N = 8 * C; a.K = C; a.A = tok; a.W = pk + o.w1; a.bias = F32(o.b1); a.h = nullptr; a.out = big;
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
        a.epilogue = NMM_EPI_RESIDUAL; a.N = C; a.K = 4 * C; a.A = big; a.W = pk + o.w2; a.bias = F32(o.b2); a.h = h; a.out = nullptr; a.no_h_store = 0;
        if (l == g.layers - 1 && g.dtype != NMM_F32) { a.out = tok; a.no_h_store = 1; }     // the sum is consumed once, by proj_out, as a bf16 operand
        if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
        a.no_h_store = 0;
    }
    // y = proj_out(h) back in NCHW + x, stored as [B, F, C, H, W]                         :130-144
    a.epilogue = NMM_EPI_OUTPUT; a.N = C; a.K = C; a.A = (g.dtype != NMM_F32) ? (const void *)tok : (const void *)h;
    a.W = pk + L.w_out; a.bias = F32(L.b_out); a.h = nullptr; a.out = nullptr; a.x = x; a.y = y;
    // N1: the GroupNorm sums of y for the motion module that consumes it next (unet_blocks.py:409-411) -- emitted by this epilogue
    // (bf16 vector path; per 32-row block and channel, then one warp per (image, group) in a fixed order: no atomics), else one pass over y
    float2 *stat_part = (float2 *)(ws + w.stat_part);
    const bool emit = y_sums != nullptr && g.dtype == NMM_BF16 && output_vec_ok(a);
    a.y_part = emit ? stat_part : nullptr;
    if ((rc = linear_dispatch(g.dtype, a, st)) != NMM_OK) return rc;
    if (emit) return launch_y_sums_channels(stat_part, y_sums, g.B * g.F, g.C, g.P, st);
    if (y_sums != nullptr) {
        nmm_shape sy = *bs;
        sy.x_stride_b = bs->y_stride_b; sy.x_stride_c = bs->y_stride_c; sy.x_stride_f = bs->y_stride_f;
        if ((rc = launch_gn_stats(g, &sy, y, gn_partial, st)) != NMM_OK) return rc;
        return launch_gn_partial_to_sums(g, gn_partial, y_sums, st);
    }
    return NMM_OK;
}

int nmm_spatial_forward(const nmm_spatial_shape *s, const void *x, const void *encoder_hidden_states, void *y, const void *packed, size_t packed_bytes,
                        void *workspace, size_t workspace_bytes, void *stream) {
    return spatial_forward_impl(s, x, encoder_hidden_states, y, packed, packed_bytes, workspace, workspace_bytes, nullptr, stream);
}

int nmm_spatial_forward_stats(const nmm_spatial_shape *s, const void *x, const void *encoder_hidden_states, void *y, const void *packed,
                              size_t packed_bytes, void *workspace, size_t workspace_bytes, double *y_sums, void *stream) {
    if (y_sums != nullptr && !aligned(y_sums, 16)) return fail(NMM_ERR_BAD_ARG, "y_sums must be 16-byte aligned");
    return spatial_forward_impl(s, x, encoder_hidden_states, y, packed, packed_bytes, workspace, workspace_bytes, y_sums, stream);
}

}  // extern "C"

/*
 * neurons_mm.h -- C ABI of libneurons_mm.so: the B200 (sm_100a) implementation of the AnimateDiff
 * motion-module forward that NEURONS' video-reconstruction stage runs 28x per denoising step.
 *
 * The reference has NO native boundary for this path (it is pure Python on PyTorch); the interface
 * replaced is the Python call
 *     VanillaTemporalModule.forward(input_tensor[b,c,f,h,w], temb, encoder_hidden_states)
 *         /root/reference/animatediff/models/motion_module.py:77-82  (-> :134-158, :210-222, :270-329)
 * made from the five UNet block classes at animatediff/models/unet_blocks.py:275,411,511,661,754.
 * Every entry point below cites the reference lines whose arithmetic it carries out.
 *
 * Conventions
 *   - plain C, no torch / CUDA types: device pointers are `void*`, the stream is a `cudaStream_t`
 *     passed as `void*` (0 = legacy default stream).
 *   - every device pointer is BORROWED from the caller (PyTorch's caching allocator); the library
 *     never allocates or frees device memory and never synchronises: all work is enqueued on the
 *     caller's stream and is CUDA-graph capturable.
 *   - every function returns NMM_OK (0) or a negative nmm_status; nmm_last_error() gives the text
 *     (thread-local).  Nothing throws or exits across the ABI.  There is no CPU fallback: on a
 *     machine without an sm_100 GPU the compute entry points return NMM_ERR_DEVICE.
 *   - token order used by all intermediate buffers: n = (b*F + f)*P + p,  P = H*W  (the reference's
 *     own "(b f) d c" order, motion_module.py:144), rows of C contiguous channels.
 */
#ifndef NEURONS_MM_H
#define NEURONS_MM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NMM_ABI_VERSION 3
#if defined(__GNUC__)
#define NMM_API __attribute__((visibility("default")))
#else
#define NMM_API
#endif
#define NMM_MAX_LAYERS 4        /* num_transformer_block; 1 in every NEURONS config (inference-v3.yaml:10) */
#define NMM_MAX_ATTN 4          /* len(attention_block_types); 2 in the UNet, 1 in SparseCtrl */
#define NMM_MAX_FRAMES 32       /* temporal_position_encoding_max_len is 24 (UNet) / 32 (SparseCtrl) */
#define NMM_GN_GROUPS 32        /* motion_module.py:95,109 */

typedef enum nmm_status {
    NMM_OK = 0,
    NMM_ERR_BAD_ARG = -1,       /* null pointer, non-positive size, misaligned pointer               */
    NMM_ERR_UNSUPPORTED = -2,   /* configuration the reference supports but this library does not    */
    NMM_ERR_WORKSPACE = -3,     /* workspace / packed-weight buffer too small                         */
    NMM_ERR_CUDA = -4,          /* a CUDA runtime call failed (text in nmm_last_error)                */
    NMM_ERR_DEVICE = -5         /* no CUDA device, or the device is not sm_100                        */
} nmm_status;

typedef enum nmm_dtype {
    NMM_F32 = 0,                /* parity mode: fp32 storage, fp32 FMA arithmetic (bar: max-abs 1e-4) */
    NMM_BF16 = 1,               /* production mode: bf16 storage + tcgen05 bf16 MMA, fp32 accumulate,
                                   fp32 residual stream, norms / softmax in fp32 (bar: max-abs 2e-2)  */
    NMM_F32X3 = 2,              /* fp32 storage (x, y, source parameters: float), fp32-grade arithmetic on the tensor cores:
                                   every Linear runs as three bf16 tcgen05 MMAs per product -- hi.hi + hi.lo + lo.hi of
                                   the two-term bf16 splits of both operands, fp32 accumulation in TMEM (bar: max-abs 1e-4,
                                   like NMM_F32, which stays as the FMA-pipe checker).  Needs channels % 64 == 0.
                                   nmm_shape.dtype only; nmm_params.dtype stays the source element type.              */
    NMM_F32X6 = 3               /* fp32 storage (x, y, source parameters: float), fp32-exact arithmetic on the tensor cores:
                                   GEMM operands are bf16 [rows, 3K] = hi | mid | lo planes (hi = bf16(v), mid = bf16(v - hi),
                                   lo = bf16(v - hi - mid): ~24 significant bits), every Linear runs as six bf16 tcgen05 MMAs per
                                   product -- the cross products of weight >= 2^-16 (lo.hi, mid.mid, hi.lo, mid.hi, hi.mid,
                                   hi.hi; the dropped terms are <= 2^-24 relative), fp32 accumulation in TMEM restarted every
                                   K = 320 with the partial sums added in fp32 by the epilogue; the spatial attention likewise
                                   (six mma.sync products for S and for O, each 32-key tile's P.V folded into O in fp32).  Measured
                                   (B200): GEMM error flat in K (1.5-2e-6 on N(0,1) outputs up to K = 5120, FMA GEMM 3.9e-6 ..
                                   1.6e-5); attention 1.5-3e-5 against fp64 at max |logit| 60 like the FMA kernels (x3: 2-2.7e-4),
                                   up to 2.7x the FMA kernels' error at smaller logits; module outputs within 2x of NMM_F32.  Needs channels % 64 == 0 (and ctx_dim % 64 == 0 for the spatial
                                   transformer).  nmm_shape.dtype only; nmm_params.dtype stays the source element type.       */
} nmm_dtype;

/* Shape + hyper-parameters of one module call.  Mirrors the arguments that reach
 * VanillaTemporalModule.__init__ (motion_module.py:49-60) and the runtime tensor geometry. */
typedef struct nmm_shape {
    int32_t batch, channels, frames, height, width;     /* logical x: [b, c, f, h, w]                 */
    int32_t heads;              /* num_attention_heads (8)                                             */
    int32_t layers;             /* num_transformer_block                                               */
    int32_t attn_blocks;        /* number of "Temporal_Self" attention blocks per transformer block    */
    int32_t pos_enc;            /* temporal_position_encoding (0/1)                                    */
    int32_t max_len;            /* temporal_position_encoding_max_len; frames <= max_len is required   */
    int32_t dtype;              /* nmm_dtype of x, y and of the arithmetic mode                        */
    float eps_gn;               /* 1e-6, motion_module.py:109                                          */
    float eps_ln;               /* 1e-5, nn.LayerNorm default (motion_module.py:201,207)               */
    int32_t ln_fold;            /* bf16 mode only: 1 = LayerNorm folded into the consuming GEMM (the producing GEMM emits
                                   row statistics + a bf16 copy of the residual; QKV / GEGLU run on gamma-folded weights and
                                   apply rstd*(acc - mean*g) + c (+ pe.W^T) in their epilogue): 3 kernels and one fp32 read of
                                   the residual stream fewer per block.  0 = separate LayerNorm kernel.  Must be the same in
                                   nmm_pack_params and nmm_forward (it changes the packed layout).                          */
    /* element strides of x and y for the b, c and f axes; (h, w) must be dense (stride W, 1).
     * x may be the contiguous "b c f h w" tensor or the [B,F,C,H,W]-storage view every UNet call site
     * passes (SURVEY 3.3); y is normally [B,F,C,H,W] storage like the reference's (motion_module.py:153-156). */
    int64_t x_stride_b, x_stride_c, x_stride_f;
    int64_t y_stride_b, y_stride_c, y_stride_f;
} nmm_shape;

/* Source parameters exactly as they sit in the nn.Module / checkpoint ("motion_modules.*" keys,
 * animatediff/utils/util.py:107-121).  All pointers are device pointers of element type `dtype`
 * (NMM_F32 or NMM_BF16), row-major [out_features, in_features] for weights. */
typedef struct nmm_attn_params {
    const void *norm_w, *norm_b;        /* transformer_blocks.L.norms.I.{weight,bias}        [C]      */
    const void *to_q, *to_k, *to_v;     /* ...attention_blocks.I.to_{q,k,v}.weight           [C,C]    */
    const void *to_out_w, *to_out_b;    /* ...attention_blocks.I.to_out.0.{weight,bias}      [C,C],[C]*/
    const void *pe;                     /* ...attention_blocks.I.pos_encoder.pe  [max_len,C] or NULL
                                           (non-persistent buffer, motion_module.py:234-239)          */
} nmm_attn_params;

typedef struct nmm_layer_params {
    nmm_attn_params attn[NMM_MAX_ATTN];
    const void *ff_norm_w, *ff_norm_b;  /* ff_norm.{weight,bias}                             [C]      */
    const void *ff_proj_w, *ff_proj_b;  /* ff.net.0.proj.{weight,bias}  (GEGLU: value|gate)  [8C,C],[8C] */
    const void *ff_out_w, *ff_out_b;    /* ff.net.2.{weight,bias}                            [C,4C],[C] */
} nmm_layer_params;

typedef struct nmm_params {
    int32_t dtype;                      /* nmm_dtype of every tensor below                            */
    const void *gn_w, *gn_b;            /* temporal_transformer.norm.{weight,bias}           [C]      */
    const void *proj_in_w, *proj_in_b;  /* temporal_transformer.proj_in.{weight,bias}        [C,C],[C]*/
    nmm_layer_params layer[NMM_MAX_LAYERS];
    const void *proj_out_w, *proj_out_b;/* temporal_transformer.proj_out.{weight,bias}       [C,C],[C]*/
} nmm_params;

/* Run-time options (process-wide; development / A-B measurement switches -- every default is the production path and no option
 * changes results beyond rounding).  Initial values come from the environment variables named below, read ONCE at first use;
 * nmm_set_option overrides them.  Nothing in the launch path calls getenv. */
typedef enum nmm_option {
    NMM_OPT_FUSED_MODULE = 0,   /* 1: C = 320 calls run on the one-kernel path (fused_module.cu).  env NMM_NO_FUSED_MODULE=1 -> 0  */
    NMM_OPT_GN_FUSE = 1,        /* 1: GroupNorm applied inside proj_in's tensor-core kernel.          env NMM_NO_GN_FUSE=1 -> 0     */
    NMM_OPT_ATTN_FUSE = 2,      /* 1: temporal attention inside the QKV projection's epilogue.        env NMM_NO_ATTN_FUSE=1 -> 0   */
    NMM_OPT_WIDE_TILE = 3,      /* 1: 256 x 320 pair tiles for long-K residual GEMMs.                 env NMM_NO_WIDE_TILE=1 -> 0   */
    NMM_OPT_GEMM_CLUSTER = 4,   /* 0: planner decides; 1 / 2: force CTAs per tile.                    env NMM_GEMM_CLUSTER          */
    NMM_OPT_GEMM_BLOCK_N = 5,   /* 0: planner decides; else force the N tile.                         env NMM_GEMM_BLOCK_N          */
    NMM_OPT_CHUNK_TOKENS = 6,   /* 0: whole tensor; else tokens per position chunk (negative result). env NMM_CHUNK_TOKENS          */
    NMM_OPT_ATTN_VARIANT = 7,   /* 0: specialised mma kernel; 1: run-time-shaped mma; 2: SIMT.        env NMM_ATTN_GENERIC / _SIMT  */
    NMM_OPT_FUSED_Y_STATS = 8,  /* nmm_forward_stats on the one-kernel C = 320 path: 1 = y sums emitted from the kernel's y store; 0 (default) =
                                   a statistics pass over the (L2-resident) y, measured faster there.  env NMM_FUSED_Y_STATS          */
    NMM_OPT_FUSED_CLUSTER = 9,  /* 0: CTA pairs when the tile count is even; 1: force the single-CTA fused kernel.  env NMM_FUSED_CLUSTER */
    NMM_OPT_SPATIAL_ATTN = 10,  /* spatial self-attention (d_h 40 / 80, >= 256 keys): 0 = tcgen05 kernel (planner: two query tiles per CTA); 1 = mma.sync kernel;
                                   other values: A/B variants of the tcgen05 kernel (csrc/spatial_attention_tc.cu).  fp32 calls (NMM_F32): 30 = always the
                                   tiled FMA-pipe kernel, 31 = always the one-warp-per-query checker; other values select by size.  env NMM_SPATIAL_ATTN */
    NMM_OPT_COUNT = 11
} nmm_option;
NMM_API int nmm_set_option(int32_t option, int64_t value);
NMM_API int64_t nmm_get_option(int32_t option);

/* ---- library / device ------------------------------------------------------------------------ */
NMM_API int nmm_abi_version(void);
NMM_API const char *nmm_last_error(void);
/* NMM_OK iff the current CUDA device is compute capability 10.x. */
NMM_API int nmm_device_check(void);
/* number of kernels this library has launched in this process (bench.py's `gpu_launches` claim). */
NMM_API uint64_t nmm_launch_count(void);

/* Optional per-kernel device timing for roofline reporting: between begin and end the library brackets every kernel
 * launch with CUDA events on the launch stream (eager launches only; launches inside a stream capture are skipped).
 * nmm_profile_end synchronises on the recorded events and fills one entry per kernel (NMM_PROFILE_KERNELS entries):
 * launches, summed device ms, and the summed ALGORITHMIC flops / bytes of those launches (DESIGN.md section 4). */
#define NMM_PROFILE_KERNELS 12
typedef struct nmm_kernel_profile {
    const char *name;
    uint64_t launches;
    double total_ms;
    double flops;
    double bytes;
} nmm_kernel_profile;
NMM_API int nmm_profile_begin(void);
NMM_API int nmm_profile_end(nmm_kernel_profile *out, int32_t max_kernels);

/* ---- whole-module forward (replaces motion_module.py:77-82 -> :134-158) ----------------------- */
NMM_API int nmm_validate(const nmm_shape *s);
NMM_API int nmm_packed_params_bytes(const nmm_shape *s, size_t *out_bytes);
NMM_API int nmm_workspace_bytes(const nmm_shape *s, size_t *out_bytes);
/* Convert + re-lay-out the module's parameters once (QKV concatenated, GEGLU value/gate rows
 * interleaved in groups of four, GEMM operands in the arithmetic dtype, biases / norm affines / PE in fp32). */
NMM_API int nmm_pack_params(const nmm_shape *s, const nmm_params *src, void *packed, size_t packed_bytes, void *stream);
/* y = module(x).  x, y: element type s->dtype with the strides in *s.  x and y must not alias.
 * `packed_bytes` must equal nmm_packed_params_bytes(s): a buffer packed for another dtype / ln_fold / geometry selects another
 * layout and is refused instead of being read out of bounds.
 * Replaces VanillaTemporalModule.forward, animatediff/models/motion_module.py:77-82 (-> :134-158, :210-222, :270-329).
 * bf16, C = 320, 8 heads, 8 or 16 frames, H*W % (128 / frames) == 0: GroupNorm statistics + ONE fused kernel for the rest
 * (csrc/fused_module.cu); other shapes: the multi-kernel pipeline (csrc/api.cu). */
NMM_API int nmm_forward(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace,
                size_t workspace_bytes, void *stream);
/* The 64-byte header nmm_pack_params writes at the start of a packed buffer for this geometry (magic, ABI, dtype, ln_fold, C, heads,
 * layers, attention blocks, max_len, pos_enc, total bytes): lets a host check what a buffer was packed for. */
NMM_API int nmm_packed_header(const nmm_shape *s, void *out, size_t out_bytes);
/* Test hook of the fused C = 320 kernel: nmm_forward plus an fp32 [N, C] snapshot (token order n = (b*F + f)*P + p) of the residual
 * stream after stage `stage_id`: 0 = proj_in (motion_module.py:145), 1 + i = attention block i (:213-217), 1 + A = feed-forward (:219).
 * NMM_ERR_UNSUPPORTED when the call would not run on the fused kernel. */
NMM_API int nmm_forward_stage(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace,
                size_t workspace_bytes, int32_t stage_id, float *stage_out, void *stream);

/* ---- per-stage entry points (kernel-level parity tests and micro-benchmarks) ------------------- */
/* GroupNorm(32, C, eps_gn) statistics per (b, f, group): motion_module.py:142.  mean/rstd: fp32 [B*F*32]. */
NMM_API int nmm_groupnorm_stats(const nmm_shape *s, const void *x, float *mean, float *rstd, void *workspace,
                        size_t workspace_bytes, void *stream);
/* GroupNorm apply fused with "(b f) c h w -> (b f) (h w) c": motion_module.py:142-144.
 * tokens: [N, C] of s->dtype.  gn_w/gn_b: fp32 [C]. */
NMM_API int nmm_groupnorm_tokens(const nmm_shape *s, const void *x, const float *gn_w, const float *gn_b, void *tokens,
                         void *workspace, size_t workspace_bytes, void *stream);
/* GroupNorm + re-layout + proj_in in ONE tensor-core kernel (bf16 only): motion_module.py:142-145.
 * h_out[N, C_out] fp32 = GroupNorm(x) as tokens . W^T + bias.  The A tiles are TMA-loaded straight from x (channel rows of positions,
 * an M-major operand) and normalised in shared memory, so the token tensor is never materialised.  W: [C_out, C] bf16; bias: fp32 [C_out]
 * or NULL.  Needs H*W % 64 == 0, N % 128 == 0, 16-byte aligned x / strides; otherwise NMM_ERR_UNSUPPORTED (use
 * nmm_groupnorm_tokens + nmm_linear; nmm_forward picks automatically). */
NMM_API int nmm_groupnorm_linear(const nmm_shape *s, const void *x, const float *gn_w, const float *gn_b, const void *W, int32_t c_out,
                         const float *bias, float *h_out, void *workspace, size_t workspace_bytes, void *stream);
/* InflatedGroupNorm(32 groups, eps_gn) of a [b, c, f, h, w] tensor, optionally followed by SiLU, written in the layout the y strides
 * describe: the norm1 / norm2 (+ nonlinearity) of ResnetBlock3D either side of the motion module (SURVEY 8(f) N1;
 * animatediff/models/resnet.py:21-29,182-198).  Only batch, channels, frames, height, width, dtype, eps_gn and the strides of *s are
 * used.  gn_w / gn_b: fp32 [C].  workspace: nmm_groupnorm_workspace_bytes(s), 256-byte aligned.  x and y must not alias. */
NMM_API int nmm_groupnorm_workspace_bytes(const nmm_shape *s, size_t *bytes);
NMM_API int nmm_inflated_groupnorm(const nmm_shape *s, const void *x, void *y, const float *gn_w, const float *gn_b, int32_t silu,
                           void *workspace, size_t workspace_bytes, void *stream);
/* GroupNorm statistics carried between neighbours instead of being recomputed (SURVEY 8(f) N1; call order unet_blocks.py:407-411:
 * resnet -> attn -> motion_module -> next resnet, whose norm1 -- resnet.py:182-198 -- normalises the motion module's output).
 * "sums" = fp64 [B*F*32][2]: (sum, sum of squares) of a [b, c, f, h, w] tensor per (b, f, GroupNorm group), 16-byte aligned.
 *   nmm_forward_stats             nmm_forward with x_sums (optional in: statistics of x -- the module's own GroupNorm skips its pass
 *                                 over x) and y_sums (optional out: statistics of y as stored, emitted from the last kernel's epilogue
 *                                 in bf16 mode -- proj_out / the fused module's y store -- and reduced without atomics, in a fixed order;
 *                                 other modes run one statistics pass over y).  Either pointer may be NULL.
 *   nmm_inflated_groupnorm_sums   nmm_inflated_groupnorm with the statistics of x handed over: one pass over x instead of two.
 *   nmm_groupnorm_sums            the statistics of any tensor in this format (workspace: nmm_groupnorm_workspace_bytes). */
NMM_API int nmm_forward_stats(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace,
                              size_t workspace_bytes, const double *x_sums, double *y_sums, void *stream);
NMM_API int nmm_inflated_groupnorm_sums(const nmm_shape *s, const void *x, void *y, const float *gn_w, const float *gn_b, int32_t silu,
                                        const double *x_sums, void *workspace, size_t workspace_bytes, void *stream);
NMM_API int nmm_groupnorm_sums(const nmm_shape *s, const void *x, double *sums, void *workspace, size_t workspace_bytes, void *stream);
/* Denoise-loop glue (SURVEY 8(f) N2): classifier-free guidance + one deterministic DDIM update in a single elementwise kernel,
 * pipeline_neuroclips.py:478-483 + DDIMScheduler.step (eta = 0, epsilon prediction, clip_sample = false):
 *   eps = eps_uncond + guidance * (eps_cond - eps_uncond)            (eps_cond == NULL: eps = eps_uncond, guidance ignored)
 *   latents = sqrt(a_prev) * (latents - sqrt(1 - a_t) * eps) / sqrt(a_t) + sqrt(1 - a_prev) * eps        (in place)
 * n elements of `dtype` (NMM_F32 / NMM_BF16), fp32 arithmetic; alpha_t / alpha_prev = alphas_cumprod at t and at the previous step. */
NMM_API int nmm_cfg_ddim_step(int32_t dtype, int64_t n, void *latents, const void *eps_uncond, const void *eps_cond, float guidance,
                      double alpha_t, double alpha_prev, void *stream);
/* LayerNorm(C, eps_ln) (+ sinusoidal PE of the token's frame): motion_module.py:212 + :277-278 (pe != NULL)
 * or :219 (pe == NULL).  h: fp32 [N,C]; out: [N,C] of s->dtype; w,b: fp32 [C]; pe: fp32 [max_len,C]. */
NMM_API int nmm_layernorm_pe(const nmm_shape *s, const float *h, const float *w, const float *b, const float *pe,
                     void *out, void *stream);
/* softmax(q k^T / sqrt(d_h)) v per (b, p, head) over the frame axis: motion_module_new.py:258-287 with the
 * head split/merge of :181-193 folded into the indexing.  qkv: [N,3C] (q|k|v), ctx: [N,C], both s->dtype. */
NMM_API int nmm_temporal_attention(const nmm_shape *s, const void *qkv, void *ctx, void *stream);

typedef enum nmm_epilogue {
    NMM_EPI_STORE = 0,          /* acc (+ bias) -> `h` (fp32 [M,N]) if non-NULL and/or `out` ([M,N] of dtype) if non-NULL */
    NMM_EPI_RESIDUAL = 1,       /* out == NULL: h = acc + bias + h (fp32, in place)   motion_module.py:213-219;
                                   out != NULL: out = acc + bias + h in `dtype`, h is only read (the last
                                   feed-forward: its sum is consumed once, by proj_out)                        */
    NMM_EPI_GEGLU = 2,          /* out[:, 2q+i] = (acc[4q+i]+b[4q+i]) * gelu_erf(acc[4q+2+i]+b[4q+2+i]), i = 0,1 -> out [M,N/2];
                                   W rows (and bias) pre-interleaved in groups of four: value 2q, value 2q+1, gate 2q, gate 2q+1
                                   (N % 4 == 0)                          motion_module_new.py:516-518          */
    NMM_EPI_OUTPUT = 3          /* y[b,c,f,p] = acc + bias + x[b,c,f,p]   motion_module.py:152-156             */
} nmm_epilogue;

/* QKV projection with the temporal attention fused into its epilogue (bf16; d_h in {40, 80}; frames in {8, 16};
 * H*W % (128 / frames) == 0): ctx = attention(tokens . Wq^T, tokens . Wk^T, tokens . Wv^T) -- motion_module.py:289-321 with
 * motion_module_new.py:258-287.  tokens: [N, C]; wqkv: [3C, C] rows of to_q, then to_k, then to_v; w_scratch: 3C*C elements (receives the
 * tile-ordered copy the kernel consumes); ctx: [N, C].  Otherwise NMM_ERR_UNSUPPORTED (use nmm_linear + nmm_temporal_attention;
 * nmm_forward picks automatically). */
NMM_API int nmm_qkv_attention(const nmm_shape *s, const void *tokens, const void *wqkv, void *w_scratch, void *ctx, void *stream);
/* D[M,N] = A[M,K] . W[N,K]^T with a fused epilogue.  A, W, out: element type `dtype` (NMM_BF16 runs on
 * tcgen05 tensor cores with fp32 accumulation in TMEM; NMM_F32 runs on fp32 FMA).  bias: fp32 [N] or NULL.
 * M = s->batch*frames*height*width is implied by `s` for NMM_EPI_OUTPUT; otherwise M is explicit. */
NMM_API int nmm_linear(int32_t dtype, int32_t epilogue, int64_t M, int32_t N, int32_t K, const void *A, const void *W,
               const float *bias, float *h, void *out, const nmm_shape *s, const void *x, void *y, void *stream);

/* ---- spatial transformer: the neighbour of the motion module inside every CrossAttn block (SURVEY 8(f) N3) ------------------------
 * Replaces Transformer3DModel.forward, /root/reference/animatediff/models/attention.py:95-148 (-> BasicTransformerBlock.forward
 * :258-300; CrossAttention / FeedForward / GEGLU arithmetic: motion_module_new.py:119-339,429-534), in the configuration every NEURONS
 * UNet / ControlNet uses (unet_blocks.py:222-237 etc.): GroupNorm(32, eps 1e-6), 1x1-convolution proj_in / proj_out
 * (use_linear_projection = False; a Linear [C, C] weight is accepted as well -- same GEMM), LayerNorm norm1/2/3, attn1 = self-attention
 * over the H*W positions of each frame, attn2 = cross-attention onto encoder_hidden_states [b, ctx_len, ctx_dim] (shared by the frames
 * of a clip, attention.py:101), GEGLU feed-forward, no attention bias / mask, no cross-frame or temporal attention inside the block.
 * Called from unet_blocks.py:273,409,509,752 immediately BEFORE the motion module of the same block; y has the [B, F, C, H, W]
 * storage of attention.py:144, which is exactly what nmm_forward then takes as a view.                                              */
typedef struct nmm_spatial_shape {
    nmm_shape base;             /* batch, channels, frames, height, width, heads (attention_head_dim = channels / heads in {40, 80, 160}),
                                   layers (num_layers), dtype (NMM_BF16 or NMM_F32), eps_gn, eps_ln, x / y strides;
                                   attn_blocks, pos_enc, max_len, ln_fold are ignored                                                  */
    int32_t ctx_len;            /* encoder_hidden_states tokens (77 CLIP tokens)                                                       */
    int32_t ctx_dim;            /* cross_attention_dim (768)                                                                           */
} nmm_spatial_shape;

typedef struct nmm_spatial_layer_params {           /* transformer_blocks.L.* (attention.py:151-236)                                  */
    const void *norm1_w, *norm1_b;                  /* norm1.{weight,bias}                         [C]                                */
    const void *attn1_q, *attn1_k, *attn1_v;        /* attn1.to_{q,k,v}.weight                     [C,C]                              */
    const void *attn1_out_w, *attn1_out_b;          /* attn1.to_out.0.{weight,bias}                [C,C],[C]                          */
    const void *norm2_w, *norm2_b;                  /* norm2.{weight,bias}                         [C]                                */
    const void *attn2_q;                            /* attn2.to_q.weight                           [C,C]                              */
    const void *attn2_k, *attn2_v;                  /* attn2.to_{k,v}.weight                       [C,ctx_dim]                        */
    const void *attn2_out_w, *attn2_out_b;          /* attn2.to_out.0.{weight,bias}                [C,C],[C]                          */
    const void *norm3_w, *norm3_b;                  /* norm3.{weight,bias}                         [C]                                */
    const void *ff_proj_w, *ff_proj_b;              /* ff.net.0.proj.{weight,bias}  (value | gate) [8C,C],[8C]                        */
    const void *ff_out_w, *ff_out_b;                /* ff.net.2.{weight,bias}                      [C,4C],[C]                         */
} nmm_spatial_layer_params;

typedef struct nmm_spatial_params {
    int32_t dtype;                                  /* NMM_F32 or NMM_BF16: element type of every tensor below                        */
    const void *gn_w, *gn_b;                        /* norm.{weight,bias}                          [C]                                */
    const void *proj_in_w, *proj_in_b;              /* proj_in.{weight,bias}                       [C,C(,1,1)],[C]                    */
    nmm_spatial_layer_params layer[NMM_MAX_LAYERS];
    const void *proj_out_w, *proj_out_b;            /* proj_out.{weight,bias}                      [C,C(,1,1)],[C]                    */
} nmm_spatial_params;

NMM_API int nmm_spatial_packed_params_bytes(const nmm_spatial_shape *s, size_t *out_bytes);
NMM_API int nmm_spatial_workspace_bytes(const nmm_spatial_shape *s, size_t *out_bytes);
NMM_API int nmm_spatial_pack_params(const nmm_spatial_shape *s, const nmm_spatial_params *src, void *packed, size_t packed_bytes, void *stream);
/* y = Transformer3DModel(x, encoder_hidden_states).sample.  x, y: element type s->base.dtype with the strides in s->base (x is normally the
 * contiguous "b c f h w" output of ResnetBlock3D; y [B,F,C,H,W] storage); encoder_hidden_states: contiguous [batch, ctx_len, ctx_dim] of the
 * same element type.  Same ownership / stream / graph-capture rules as nmm_forward. */
NMM_API int nmm_spatial_forward(const nmm_spatial_shape *s, const void *x, const void *encoder_hidden_states, void *y, const void *packed,
                                size_t packed_bytes, void *workspace, size_t workspace_bytes, void *stream);
/* nmm_spatial_forward that also emits the GroupNorm sums of y ("sums" format of nmm_forward_stats: fp64 [B*F*32][2]) from proj_out's
 * epilogue: the motion module called next on y (unet_blocks.py:409-411) takes them as x_sums and skips its statistics pass over y --
 * SURVEY 8(f) N1 with the real producer.  y_sums may be NULL. */
NMM_API int nmm_spatial_forward_stats(const nmm_spatial_shape *s, const void *x, const void *encoder_hidden_states, void *y, const void *packed,
                                      size_t packed_bytes, void *workspace, size_t workspace_bytes, double *y_sums, void *stream);
/* softmax(q k^T / sqrt(head_dim)) v per (image, head), flash-style (scores never materialised): CrossAttention._attention,
 * motion_module_new.py:258-287, with the head split / merge of :181-193 folded into the indexing.  q: `images` x [q_len rows] of
 * heads * head_dim channels at the given row / image strides (elements); k, v: [kv_len rows] per kv image, kv image of q image i =
 * i / kv_div (kv_div = frames for the text cross-attention, 1 for self-attention); o like q.  dtype NMM_BF16 (tensor cores; 16-byte
 * aligned, strides % 8 == 0), NMM_F32 (fp32 checker kernel) or NMM_F32X3 (fp32-grade, 3 bf16 MMAs per product): q, k, v are then
 * bf16 rows of a hi plane and a lo plane, the lo plane half a row stride after the hi plane (e.g. q rows [hi q | lo q], k | v rows
 * [hi k | hi v | lo k | lo v]), o is fp32.  NMM_F32X6 (fp32-exact, 6 bf16 MMAs per product): q, k, v are bf16 rows of hi | mid | lo planes,
 * each plane a third of a row stride after the previous one; o is fp32.  head_dim in {40, 80, 160}. */
NMM_API int nmm_spatial_attention(int32_t dtype, const void *q, const void *k, const void *v, void *o, int64_t q_row_stride, int64_t kv_row_stride,
                                  int64_t o_row_stride, int64_t q_image_stride, int64_t kv_image_stride, int64_t o_image_stride, int32_t q_len,
                                  int32_t kv_len, int32_t heads, int32_t head_dim, int32_t images, int32_t kv_div, void *stream);

/* ---- temporal attention of the blurry-video decoder (SURVEY 8(f) N4) -----------------------------------------------------------------
 * Replaces the `temp_attn` + blend lines of AttnUpDecoderBlock2D.forward / UNetMidBlock2D.forward,
 * /root/reference/model_variants/video_decoder.py:237-248 and :394-406:
 *     y = weight * x + (1 - weight) * rearrange(temp_attn(rearrange(x, '(b t) c h w -> (b h w) t c')), '... -> (b t) c h w')
 * with temp_attn = diffusers' Attention(c, heads = c / dim_head, norm_num_groups = 32, eps, residual_connection = True, bias = True,
 * rescale_output_factor, _from_deprecated_attn_block = True) (video_decoder.py:204-216,353-365; class imported from the un-vendored
 * `diffusers.models.attention_processor`).  PARITY UNPINNED: the class cannot be imported here, its arithmetic is restated
 * (oracle/decoder_oracle.py).  x, y: [(b t), c, h, w] = a [b, c, t, h, w] tensor in [B, F, C, H, W] storage, described by nmm_shape with
 * frames = t, heads = c / dim_head, eps_gn = the block's resnet_eps (1e-6), dtype NMM_F32 or NMM_BF16; layers / attn_blocks / pos_enc /
 * max_len / ln_fold are ignored. */
typedef struct nmm_decoder_attn_params {
    int32_t dtype;                                  /* NMM_F32 or NMM_BF16: element type of every tensor below              */
    const void *gn_w, *gn_b;                        /* temp_attn.group_norm.{weight,bias}        [C]                        */
    const void *to_q_w, *to_q_b;                    /* temp_attn.to_q.{weight,bias}              [C,C],[C]                  */
    const void *to_k_w, *to_k_b, *to_v_w, *to_v_b;  /* temp_attn.to_k / to_v                                                */
    const void *to_out_w, *to_out_b;                /* temp_attn.to_out.0.{weight,bias}          [C,C],[C]                  */
} nmm_decoder_attn_params;
NMM_API int nmm_decoder_attn_packed_bytes(int32_t channels, int32_t dtype, size_t *out_bytes);
NMM_API int nmm_decoder_attn_workspace_bytes(const nmm_shape *s, size_t *out_bytes);
/* blend_weight = the block's scalar `weights[i]` (video_decoder.py:217,366; folded into the output projection at pack time: re-pack when
 * it changes); rescale_output_factor must be 1 (it is in every block of DecoderVideo), otherwise NMM_ERR_UNSUPPORTED. */
NMM_API int nmm_decoder_attn_pack(int32_t channels, int32_t dtype, const nmm_decoder_attn_params *src, float blend_weight,
                                  float rescale_output_factor, void *packed, size_t packed_bytes, void *stream);
NMM_API int nmm_decoder_temporal_attention(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace,
                                           size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NEURONS_MM_H */

// C ABI of libneurons_mm.so (include/neurons_mm.h): validation, parameter packing, workspace carving and the
// kernel sequence of one VanillaTemporalModule.forward (motion_module.py:77-82 -> :134-158 -> :210-222 -> :270-329).
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"
#include "epilogue.cuh"

namespace nmm {

std::atomic<uint64_t> g_launches{0};

std::string &last_error_ref() {
    static thread_local std::string s;
    return s;
}
int fail(int status, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    return status;
}

// ---- run-time options ------------------------------------------------------------------------------------------
namespace {
std::atomic<int64_t> g_opts[NMM_OPT_COUNT];
std::once_flag g_opts_once;
void init_opts() {
    auto flag_off = [](const char *name) { const char *e = getenv(name); return (e && *e && strcmp(e, "0") != 0) ? 0 : 1; };
    auto num = [](const char *name) { const char *e = getenv(name); return e ? atoll(e) : 0ll; };
    g_opts[NMM_OPT_FUSED_MODULE] = flag_off("NMM_NO_FUSED_MODULE");
    g_opts[NMM_OPT_GN_FUSE] = flag_off("NMM_NO_GN_FUSE");
    g_opts[NMM_OPT_ATTN_FUSE] = flag_off("NMM_NO_ATTN_FUSE");
    g_opts[NMM_OPT_WIDE_TILE] = flag_off("NMM_NO_WIDE_TILE");
    g_opts[NMM_OPT_GEMM_CLUSTER] = num("NMM_GEMM_CLUSTER");
    g_opts[NMM_OPT_GEMM_BLOCK_N] = num("NMM_GEMM_BLOCK_N");
    g_opts[NMM_OPT_CHUNK_TOKENS] = num("NMM_CHUNK_TOKENS");
    g_opts[NMM_OPT_ATTN_VARIANT] = getenv("NMM_ATTN_SIMT") ? 2 : getenv("NMM_ATTN_GENERIC") ? 1 : 0;
    g_opts[NMM_OPT_FUSED_Y_STATS] = num("NMM_FUSED_Y_STATS");
    g_opts[NMM_OPT_FUSED_CLUSTER] = num("NMM_FUSED_CLUSTER");
    g_opts[NMM_OPT_SPATIAL_ATTN] = num("NMM_SPATIAL_ATTN");
}
}  // namespace
int64_t opt(int option) {
    std::call_once(g_opts_once, init_opts);
    return (option >= 0 && option < NMM_OPT_COUNT) ? g_opts[option].load(std::memory_order_relaxed) : 0;
}

// ---- per-kernel device timing ---------------------------------------------------------------------------------
namespace {
struct ProfRecord { cudaEvent_t start, stop; int kid; double flops, bytes; };
struct Profiler {
    bool enabled = false;
    std::vector<ProfRecord> rec;      // used records
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pool;   // reusable event pairs
    std::mutex mu;
} g_prof;
}  // namespace

ProfScope::ProfScope(int kid, cudaStream_t stream, double flops, double bytes) : slot(-1), st(stream) {
    if (!g_prof.enabled) return;
    std::lock_guard<std::mutex> lk(g_prof.mu);
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return;   // events cannot time inside a capture
    ProfRecord r;
    if (g_prof.pool.empty()) {
        if (cudaEventCreate(&r.start) != cudaSuccess || cudaEventCreate(&r.stop) != cudaSuccess) return;
    } else {
        r.start = g_prof.pool.back().first; r.stop = g_prof.pool.back().second; g_prof.pool.pop_back();
    }
    r.kid = kid; r.flops = flops; r.bytes = bytes;
    cudaEventRecord(r.start, stream);
    g_prof.rec.push_back(r);
    slot = (int)g_prof.rec.size() - 1;
}
ProfScope::~ProfScope() {
    if (slot < 0) return;
    std::lock_guard<std::mutex> lk(g_prof.mu);
    if (slot < (int)g_prof.rec.size()) cudaEventRecord(g_prof.rec[slot].stop, st);
}

// ---- packed parameter layout -------------------------------------------------------------------------
struct AttnOff { size_t ln_w, ln_b, wqkv, wqkv_t, wo, bo, pe, g_qkv, c_qkv, pew, wo_tail; };   // wqkv_t: tile-ordered copy (fused attention); g/c/pew: LayerNorm folding; wo_tail: fused module
struct LayerOff { AttnOff attn[NMM_MAX_ATTN]; size_t ff_ln_w, ff_ln_b, w1, b1, w2, b2, g1, c1; };
struct PackedLayout {
    size_t header, gn_w, gn_b, w_in, b_in;
    LayerOff layer[NMM_MAX_LAYERS];
    size_t w_out, b_out;
    // fused C = 320 module kernel: proj_in weight with the GroupNorm gamma folded in, its bias (+ beta . W_in^T), scratch for the fold,
    // cumulative biases, and the per-phase fp32 vector blocks (FmParams, fused_module.cu)
    size_t w_in_g, b_in_g, fold_tmp, cbias, vec_attn[NMM_MAX_ATTN], vec_ff, vec_fin;
    size_t total;
};

// First 256 bytes of every packed buffer: what it was packed for.  nmm_forward refuses a buffer whose header does not match the call
// (another dtype / head count / LayerNorm-folding mode would select another layout and read out of bounds).
struct PackedHeader { uint32_t magic, abi; int32_t dtype, ln_fold, C, heads, layers, A, max_len, pos_enc; uint64_t total; uint64_t reserved[2]; };
static_assert(sizeof(PackedHeader) == 64, "packed header is 64 bytes");
constexpr uint32_t PACKED_MAGIC = 0x4D4D4E32u;      // "2NMM"

// does this module keep a tile-ordered q|k|v weight for the fused QKV + attention kernel?  (shape-independent part of the test)
static bool attn_fuse_weights(const Geo &g) {
    return g.dtype == NMM_BF16 && !g.ln_fold && g.C % NMM_ATTN_TILE_CH == 0 && (g.dh == 40 || g.dh == 80);
}

static PackedLayout packed_layout(const Geo &g) {
    PackedLayout L;
    memset(&L, 0, sizeof(L));
    size_t off = 0;
    const size_t C = g.C, ws = operand_size(g.dtype);
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    L.header = take(sizeof(PackedHeader));
    L.gn_w = take(C * 4); L.gn_b = take(C * 4);
    L.w_in = take(C * C * ws); L.b_in = take(C * 4);
    for (int l = 0; l < g.layers; l++) {
        for (int i = 0; i < g.A; i++) {
            AttnOff &a = L.layer[l].attn[i];
            a.ln_w = take(C * 4); a.ln_b = take(C * 4);
            a.wqkv = take(3 * C * C * ws); a.wo = take(C * C * ws); a.bo = take(C * 4);
            a.wqkv_t = take(attn_fuse_weights(g) ? 3 * C * C * ws : 0);
            a.pe = take(g.pos_enc ? (size_t)g.max_len * C * 4 : 0);
            a.g_qkv = take(g.ln_fold ? 3 * C * 4 : 0); a.c_qkv = take(g.ln_fold ? 3 * C * 4 : 0);
            a.pew = take(g.ln_fold && g.pos_enc ? (size_t)g.max_len * 3 * C * 4 : 0);
            a.wo_tail = take(fused_module_weights(g) ? (size_t)4 * C * 16 * ws : 0);      // 16 of every 80 to_out input channels
        }
        LayerOff &lo = L.layer[l];
        lo.ff_ln_w = take(C * 4); lo.ff_ln_b = take(C * 4);
        lo.w1 = take(8 * C * C * ws); lo.b1 = take(8 * C * 4);
        lo.w2 = take(4 * C * C * ws); lo.b2 = take(C * 4);
        lo.g1 = take(g.ln_fold ? 8 * C * 4 : 0); lo.c1 = take(g.ln_fold ? 8 * C * 4 : 0);
    }
    L.w_out = take(C * C * ws); L.b_out = take(C * 4);
    {
        const bool fm = fused_module_weights(g);
        const size_t rows = g.pos_enc ? (size_t)g.max_len : 1;
        L.w_in_g = take(fm ? C * C * ws : 0); L.b_in_g = take(fm ? C * 4 : 0); L.fold_tmp = take(fm ? C * 4 : 0);
        L.cbias = take(fm ? (size_t)(g.A + 2) * C * 4 : 0);
        for (int i = 0; i < g.A; i++) L.vec_attn[i] = take(fm ? (2 + rows) * C * 4 : 0);
        L.vec_ff = take(fm ? 3 * C * 4 : 0); L.vec_fin = take(fm ? 2 * C * 4 : 0);
    }
    L.total = off;
    return L;
}

// ---- chunked execution + workspace layout ---------------------------------------------------------------------------
// Every stage after the GroupNorm statistics is local to a spatial position (Linear / LayerNorm / GEGLU per token, attention per
// position over the frames), so the module is run chunk by chunk over position ranges [p0, p0 + pc).  With pc chosen so that a
// chunk's intermediates (tokens 2 B + residual 4 B + qkv|act 8 B + ctx 2 B per token-channel in bf16 mode) stay around 40 MB,
// they are produced and consumed inside the 126 MB L2 and the same workspace addresses are overwritten by the next chunk before
// their dirty lines are ever evicted: the intermediates never reach HBM (write bandwidth, ~3.2-3.9 TB/s on this part, is what
// bounds the unchunked pipeline).  HBM traffic per call would drop from ~116 B to ~6 B per token-channel (x twice, y once).
// Chunk-local token order: row = (b*F + f)*pc + (p - p0).   NMM_CHUNK_TOKENS=<tokens> enables it (experiment; default off).
static int chunk_positions(const Geo &g) {
    // Measured on B200 (profiles/r1_chunk_sweep.txt): chunking LOSES at every chunk size (4096 tokens: 14.2 ms/step, 16384: 8.7,
    // off: 8.0) -- the per-kernel fixed cost (launch, ramp, tail; ~10 us) outweighs the saved HBM traffic, so it is off by default.
    const int64_t target = opt(NMM_OPT_CHUNK_TOKENS);       // tokens per chunk; 0 = whole tensor
    if (target <= 0 || g.P % 64 != 0) return g.P;
    int64_t pc = target / ((int64_t)g.B * g.F) / 64 * 64;
    if (pc < 64) pc = 64;
    return pc >= g.P ? g.P : (int)pc;
}

struct WorkLayout { size_t gn_partial, tok, tok2, h, big, ctx, ln_part, stat_part, total; };
static WorkLayout work_layout(const Geo &g) {
    WorkLayout w;
    size_t off = 0;
    // es: bytes per GEMM-operand element (NMM_F32X6: three bf16 planes); the fp32 q | k | v of the fp32-grade modes fit in `big` (12 <= 4 es)
    const size_t es = operand_size(g.dtype), NC = (size_t)g.B * g.F * chunk_positions(g) * g.C;     // one chunk
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
    w.gn_partial = take(gn_partial_bytes(g));
    w.tok = take(NC * es);          // GroupNorm tokens / LayerNorm output / GEMM-dtype copy of h for proj_out
    w.h = take(NC * 4);             // fp32 residual stream
    w.big = take(NC * 4 * es);      // qkv [n,3C] and GEGLU activations [n,4C] (never live together)
    w.ctx = take(NC * es);          // attention context
    // LayerNorm folding: second token buffer (bf16 copy of the residual stream) + per-row partial statistics
    // ([n][2 * n_tiles][2] fp32, n_tiles <= C / 32)
    w.tok2 = take(g.ln_fold ? NC * es : 0);
    w.ln_part = take(g.ln_fold ? NC / 32 * 2 * 2 * 4 : 0);
    // N1: fp32 (sum, sum of squares) partials of y from the last kernel: [N / 32][C] (GEMM epilogue) or [tiles][F][32] (fused module, smaller)
    w.stat_part = take(((size_t)g.N + 31) / 32 * g.C * sizeof(float2));
    w.total = off;
    return w;
}

static int validate(const nmm_shape *s) {
    if (!s) return fail(NMM_ERR_BAD_ARG, "shape is NULL");
    if (s->batch <= 0 || s->channels <= 0 || s->frames <= 0 || s->height <= 0 || s->width <= 0)
        return fail(NMM_ERR_BAD_ARG, "non-positive dimension");
    if (s->dtype != NMM_F32 && s->dtype != NMM_BF16 && s->dtype != NMM_F32X3 && s->dtype != NMM_F32X6) return fail(NMM_ERR_BAD_ARG, "unknown dtype %d", s->dtype);
    if (s->dtype == NMM_F32X3 && s->channels % 64 != 0)
        return fail(NMM_ERR_UNSUPPORTED, "NMM_F32X3 (3 x bf16 tensor-core mode) needs channels %% 64 == 0 (got %d); use NMM_F32", s->channels);
    if (s->dtype == NMM_F32X6 && s->channels % 64 != 0)
        return fail(NMM_ERR_UNSUPPORTED, "NMM_F32X6 (6 x bf16 tensor-core mode) needs channels %% 64 == 0 (got %d); use NMM_F32", s->channels);
    if (s->channels % NMM_GN_GROUPS != 0) return fail(NMM_ERR_BAD_ARG, "channels (%d) must be divisible by %d GroupNorm groups", s->channels, NMM_GN_GROUPS);
    if (s->heads <= 0 || s->channels % s->heads != 0) return fail(NMM_ERR_BAD_ARG, "channels (%d) must be divisible by heads (%d)", s->channels, s->heads);
    if (s->layers <= 0 || s->layers > NMM_MAX_LAYERS) return fail(NMM_ERR_UNSUPPORTED, "num_transformer_block %d outside [1,%d]", s->layers, NMM_MAX_LAYERS);
    if (s->attn_blocks <= 0 || s->attn_blocks > NMM_MAX_ATTN) return fail(NMM_ERR_UNSUPPORTED, "%d attention blocks outside [1,%d]", s->attn_blocks, NMM_MAX_ATTN);
    if (s->frames > NMM_MAX_FRAMES) return fail(NMM_ERR_UNSUPPORTED, "frames %d > %d", s->frames, NMM_MAX_FRAMES);
    if (s->pos_enc && s->frames > s->max_len) return fail(NMM_ERR_BAD_ARG, "frames (%d) exceed temporal_position_encoding_max_len (%d)", s->frames, s->max_len);
    if (s->heads * s->frames > 256) return fail(NMM_ERR_UNSUPPORTED, "heads*frames > 256");
    if ((int64_t)s->batch * s->frames > 65535) return fail(NMM_ERR_UNSUPPORTED, "batch*frames > 65535");
    if ((int64_t)s->batch * s->frames * s->height * s->width * (int64_t)s->channels >= ((int64_t)1 << 40)) return fail(NMM_ERR_UNSUPPORTED, "tensor too large");
    return NMM_OK;
}

int device_check() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(NMM_ERR_DEVICE, "no CUDA device: %s", cudaGetErrorString(e)); }
    int major = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(NMM_ERR_DEVICE, "cannot query device: %s", cudaGetErrorString(e)); }
    if (major != 10) return fail(NMM_ERR_DEVICE, "device compute capability %d.x is not sm_100 (this library is B200-only)", major);
    return NMM_OK;
}

// ---- parameter packing kernels ---------------------------------------------------------------------------
// dst[r, :] = src[map(r), :] with dtype conversion.  interleave_half > 0 : GEGLU packing in groups of four rows
//   packed rows 4q .. 4q+3  =  value 2q, value 2q+1, gate 2q, gate 2q+1        (gate j = source row j + half; motion_module_new.py:516-517 chunk(2))
// so that the accumulator columns of one thread hold (v0, v1, g0, g1): register-adjacent pairs for the packed fp32x2 epilogue math.
__host__ __device__ inline int64_t geglu_src_row(int64_t r, int64_t half) {
    return half > 0 ? 2 * (r >> 2) + (r & 1) + ((r >> 1) & 1) * half : r;
}
template <typename TS, typename TD>
__global__ void convert_rows_kernel(const TS *__restrict__ src, TD *__restrict__ dst, int64_t rows, int64_t cols, int64_t half) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    const int64_t total = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        const int64_t sr = geglu_src_row(r, half);
        dst[i] = from_f32<TD>(to_f32(src[sr * cols + c]));
    }
}

// NMM_F32X3 weights: dst is bf16 [rows, 2 * cols], row r = hi plane | lo plane of src row map(r)  (w = hi + lo + O(2^-17 w));
// NMM_F32X6 (PL 3): bf16 [rows, 3 * cols], hi | mid | lo planes (w = hi + mid + lo + O(2^-24 w))
template <typename TS, int PL = 2>
__global__ void split_rows_kernel(const TS *__restrict__ src, bf16 *__restrict__ dst, int64_t rows, int64_t cols, int64_t half) {
    pdl_wait();
    pdl_launch_dependents();
    const int64_t total = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        split1_store<PL>(dst + r * PL * cols, (int)cols, (int)c, to_f32(src[geglu_src_row(r, half) * cols + c]));
    }
}

int launch_convert_rows(const void *src, int src_dtype, void *dst, int dst_dtype, int64_t rows, int64_t cols, int half, cudaStream_t st) {
    if (!src || !dst) return fail(NMM_ERR_BAD_ARG, "NULL parameter tensor");
    const int64_t total = rows * cols;
    if (total == 0) return NMM_OK;
    const int threads = 256;
    const int blocks = (int)std::min<int64_t>(ceil_div(total, threads), 148 * 16);
    ProfScope prof(K_PACK, st, 0.0, (double)total * (dtype_size(src_dtype) + operand_size(dst_dtype)));
    if (dst_dtype == NMM_F32X3) {
        if (src_dtype == NMM_F32) launch_pdl(split_rows_kernel<float>, blocks, threads, 0, st, (const float *)src, (bf16 *)dst, rows, cols, (int64_t)half);
        else if (src_dtype == NMM_BF16) launch_pdl(split_rows_kernel<bf16>, blocks, threads, 0, st, (const bf16 *)src, (bf16 *)dst, rows, cols, (int64_t)half);
        else return fail(NMM_ERR_BAD_ARG, "unknown parameter dtype");
        NMM_LAUNCHED("split_rows_kernel");
        return NMM_OK;
    }
    if (dst_dtype == NMM_F32X6) {
        if (src_dtype == NMM_F32) launch_pdl(split_rows_kernel<float, 3>, blocks, threads, 0, st, (const float *)src, (bf16 *)dst, rows, cols, (int64_t)half);
        else if (src_dtype == NMM_BF16) launch_pdl(split_rows_kernel<bf16, 3>, blocks, threads, 0, st, (const bf16 *)src, (bf16 *)dst, rows, cols, (int64_t)half);
        else return fail(NMM_ERR_BAD_ARG, "unknown parameter dtype");
        NMM_LAUNCHED("split_rows_kernel");
        return NMM_OK;
    }
    if (src_dtype == NMM_F32 && dst_dtype == NMM_F32) launch_pdl(convert_rows_kernel<float, float>, blocks, threads, 0, st, (const float *)src, (float *)dst, rows, cols, half);
    else if (src_dtype == NMM_F32 && dst_dtype == NMM_BF16) launch_pdl(convert_rows_kernel<float, bf16>, blocks, threads, 0, st, (const float *)src, (bf16 *)dst, rows, cols, half);
    else if (src_dtype == NMM_BF16 && dst_dtype == NMM_F32) launch_pdl(convert_rows_kernel<bf16, float>, blocks, threads, 0, st, (const bf16 *)src, (float *)dst, rows, cols, half);
    else if (src_dtype == NMM_BF16 && dst_dtype == NMM_BF16) launch_pdl(convert_rows_kernel<bf16, bf16>, blocks, threads, 0, st, (const bf16 *)src, (bf16 *)dst, rows, cols, half);
    else return fail(NMM_ERR_BAD_ARG, "unknown parameter dtype");
    NMM_LAUNCHED("convert_rows_kernel");
    return NMM_OK;
}

// q|k|v weight [3C, C] (rows: all of q, then k, then v) -> tile order of the fused QKV + attention kernel: for each 80-channel tile t,
// its 80 q rows, then its 80 k rows, then its 80 v rows (tile t = rows 240 t .. 240 t + 239).  bf16, 16-byte vector copy.
__global__ void qkv_tile_order_kernel(const bf16 *__restrict__ src, bf16 *__restrict__ dst, int C) {
    pdl_wait();
    pdl_launch_dependents();
    const int vec_per_row = C / 8;
    const int64_t total = (int64_t)3 * C * vec_per_row;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / vec_per_row), v = (int)(i - (int64_t)r * vec_per_row);
        const int t = r / (3 * NMM_ATTN_TILE_CH), w = r - t * 3 * NMM_ATTN_TILE_CH;
        const int seg = w / NMM_ATTN_TILE_CH, j = w - seg * NMM_ATTN_TILE_CH;
        const int sr = seg * C + t * NMM_ATTN_TILE_CH + j;
        reinterpret_cast<uint4 *>(dst)[i] = __ldg(reinterpret_cast<const uint4 *>(src) + (int64_t)sr * vec_per_row + v);
    }
}
static int launch_qkv_tile_order(const void *src, void *dst, int C, cudaStream_t st) {
    if (C % NMM_ATTN_TILE_CH != 0 || C % 8 != 0 || !aligned(src, 16) || !aligned(dst, 16)) return fail(NMM_ERR_UNSUPPORTED, "qkv tile order needs C %% 80 == 0");
    const int64_t total = (int64_t)3 * C * (C / 8);
    const int blocks = (int)std::min<int64_t>(ceil_div(total, 256), 148 * 16);
    ProfScope prof(K_PACK, st, 0.0, (double)total * 32);
    launch_pdl(qkv_tile_order_kernel, blocks, 256, 0, st, (const bf16 *)src, (bf16 *)dst, C);
    NMM_LAUNCHED("qkv_tile_order_kernel");
    return NMM_OK;
}

// ---- LayerNorm folding (pack time) -------------------------------------------------------------------------------------------
// For a Linear that consumes LayerNorm(h) (+ pe):   (LN(h) + pe) . W^T + b
//     = rstd * ( h . (gamma (.) W)^T  -  mean * g )  +  c  +  pe . W^T,      g[n] = sum_c gamma[c] W[n,c],  c[n] = sum_c beta[c] W[n,c] + b[n]
// so the GEMM can run on the RAW residual rows with the gamma-folded weight W' = bf16(gamma (.) W) and the epilogue finishes the
// normalisation.  g is summed over the bf16-ROUNDED W' (exactly what the tensor core multiplies), c and pe.W^T in fp32.
// Row mapping as in convert_rows_kernel (GEGLU interleave).
template <typename TS>
__global__ void fold_weight_kernel(const TS *__restrict__ src, const TS *__restrict__ gamma, bf16 *__restrict__ dst, int64_t rows,
                                   int64_t cols, int64_t half) {
    pdl_wait();
    pdl_launch_dependents();
    const int64_t total = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        const int64_t sr = geglu_src_row(r, half);
        dst[i] = __float2bfloat16_rn(to_f32(src[sr * cols + c]) * to_f32(gamma[c]));
    }
}
// one 128-thread CTA per output row r: g[r], c[r] and pew[f][r] (f < max_len; pew may be null)
template <typename TS>
__global__ void __launch_bounds__(128) fold_tables_kernel(const TS *__restrict__ src, const bf16 *__restrict__ folded,
                                                          const TS *__restrict__ beta, const TS *__restrict__ bias,
                                                          const TS *__restrict__ pe, float *__restrict__ g_out,
                                                          float *__restrict__ c_out, float *__restrict__ pew_out, int64_t cols,
                                                          int64_t half, int max_len, int64_t pew_pitch) {
    pdl_wait();
    pdl_launch_dependents();
    __shared__ float red[4];
    const int64_t r = blockIdx.x;
    const int64_t sr = geglu_src_row(r, half);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    auto block_sum = [&](float v) {
        v = warp_sum(v);
        __syncthreads();
        if (lane == 0) red[warp] = v;
        __syncthreads();
        return red[0] + red[1] + red[2] + red[3];
    };
    float gs = 0.f, cs = 0.f;
    for (int64_t c = threadIdx.x; c < cols; c += 128) {
        gs += to_f32(folded[r * cols + c]);
        cs = fmaf(to_f32(beta[c]), to_f32(src[sr * cols + c]), cs);
    }
    gs = block_sum(gs);
    cs = block_sum(cs);
    if (threadIdx.x == 0) { g_out[r] = gs; c_out[r] = cs + (bias ? to_f32(bias[sr]) : 0.f); }
    if (pew_out != nullptr) {
        for (int f = 0; f < max_len; f++) {
            float ps = 0.f;
            for (int64_t c = threadIdx.x; c < cols; c += 128) ps = fmaf(to_f32(pe[(int64_t)f * cols + c]), to_f32(src[sr * cols + c]), ps);
            ps = block_sum(ps);
            if (threadIdx.x == 0) pew_out[(int64_t)f * pew_pitch + r] = ps;
        }
    }
}

template <typename TS>
static int fold_linear_t(const void *w, const void *gamma, const void *beta, const void *bias, const void *pe, bf16 *dst_w, float *g_out,
                         float *c_out, float *pew_out, int64_t rows, int64_t cols, int half, int max_len, int64_t pew_pitch, cudaStream_t st) {
    if (!w || !gamma || !beta) return fail(NMM_ERR_BAD_ARG, "NULL parameter tensor");
    const int blocks = (int)std::min<int64_t>(ceil_div(rows * cols, 256), 148 * 16);
    {
        ProfScope prof(K_PACK, st, 0.0, (double)rows * cols * (sizeof(TS) + 2));
        launch_pdl(fold_weight_kernel<TS>, blocks, 256, 0, st, (const TS *)w, (const TS *)gamma, dst_w, rows, cols, (int64_t)half);
    }
    NMM_LAUNCHED("fold_weight_kernel");
    {
        ProfScope prof(K_PACK, st, 0.0, (double)rows * cols * (sizeof(TS) + 2));
        launch_pdl(fold_tables_kernel<TS>, (unsigned)rows, 128, 0, st, (const TS *)w, (const bf16 *)dst_w, (const TS *)beta, (const TS *)bias,
                   (const TS *)pe, g_out, c_out, pew_out, cols, (int64_t)half, max_len, pew_pitch);
    }
    NMM_LAUNCHED("fold_tables_kernel");
    return NMM_OK;
}
static int fold_linear(int src_dtype, const void *w, const void *gamma, const void *beta, const void *bias, const void *pe, void *dst_w,
                       float *g_out, float *c_out, float *pew_out, int64_t rows, int64_t cols, int half, int max_len, int64_t pew_pitch,
                       cudaStream_t st) {
    if (src_dtype == NMM_F32)
        return fold_linear_t<float>(w, gamma, beta, bias, pe, (bf16 *)dst_w, g_out, c_out, pew_out, rows, cols, half, max_len, pew_pitch, st);
    return fold_linear_t<bf16>(w, gamma, beta, bias, pe, (bf16 *)dst_w, g_out, c_out, pew_out, rows, cols, half, max_len, pew_pitch, st);
}

// ---- extra packed tensors of the fused C = 320 module kernel (fused_module.cu) ----------------------------------------------------
// to_out input channels 64-79 of every head pair (80 channels) as an un-swizzled K-major B operand, one contiguous 5 KB block per
// (pair, N half):  dst[hp][half][chunk 0..1][row 0..159][8] = Wo[half * 160 + row][hp * 80 + 64 + chunk * 8 + e]
__global__ void wo_tail_kernel(const bf16 *__restrict__ wo, bf16 *__restrict__ dst, int C) {
    pdl_wait();
    pdl_launch_dependents();
    const int total = 4 * 2 * 2 * 160 * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7, row = (i >> 3) % 160, chunk = (i / (8 * 160)) & 1, half = (i / (8 * 160 * 2)) & 1, hp = i / (8 * 160 * 4);
        dst[i] = wo[(size_t)(half * 160 + row) * C + hp * 80 + 64 + chunk * 8 + e];
    }
}
// cb[0] = b_in; cb[1 + i] = cb[i] + bo_i; cb[A + 1] = cb[A] + b2 (fp32, packed biases): what the readers of the TMEM-resident
// residual stream add, since the GEMMs accumulate onto it without their bias.
struct BiasList { const float *b[NMM_MAX_ATTN + 2]; int n; };
__global__ void cumulative_bias_kernel(float *__restrict__ cb, BiasList list, int C) {
    pdl_wait();
    pdl_launch_dependents();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float acc = 0.f;
    for (int k = 0; k < list.n; k++) { acc += list.b[k][c]; cb[(size_t)k * C + c] = acc; }
}
// dst = [a | b | c + d[r] for r < rows]   (vectors of C floats; c, d may be null: treated as zero; d has `rows` rows)
__global__ void vector_block_kernel(float *__restrict__ dst, const float *__restrict__ a, const float *__restrict__ b, const float *__restrict__ c,
                                    const float *__restrict__ d, int rows, int C) {
    pdl_wait();
    pdl_launch_dependents();
    const int total = (2 + rows) * C;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int r = i / C, col = i - r * C;
        float v;
        if (r == 0) v = a[col];
        else if (r == 1) v = b[col];
        else v = (c ? c[col] : 0.f) + (d ? d[(size_t)(r - 2) * C + col] : 0.f);
        dst[i] = v;
    }
}
__global__ void write_header_kernel(PackedHeader hd, PackedHeader *dst) {
    pdl_wait();
    pdl_launch_dependents();
    if (threadIdx.x == 0 && blockIdx.x == 0) *dst = hd;
}

// Sinusoidal table when the caller does not hand over the module's own `pe` buffer (motion_module.py:234-238).
__global__ void make_pe_kernel(float *__restrict__ pe, int max_len, int C) {
    pdl_wait();                    // PDL: the previous kernel has completed (no-op without the launch attribute)
    pdl_launch_dependents();       // let the next kernel's launch + prologue overlap this kernel
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= max_len * C) return;
    const int t = i / C, c = i % C;
    const float div = expf((float)(c & ~1) * (-logf(10000.0f) / (float)C));
    pe[i] = (c & 1) ? cosf((float)t * div) : sinf((float)t * div);
}

static int linear(const Geo &g, const LinearArgs &a, cudaStream_t st) {
    if (g.dtype == NMM_F32X3 || g.dtype == NMM_F32X6) {      // fp32-grade / fp32-exact on the tensor cores: operands are bf16 planes (gemm_tcgen05.cu, PL)
        LinearArgs b = a;
        b.planes = planes_of(g.dtype);
        return launch_linear_tc(b, st);
    }
    return g.dtype == NMM_BF16 ? launch_linear_tc(a, st) : launch_linear_simt(a, st);
}
int linear_dispatch(int dtype, const LinearArgs &a, cudaStream_t st) {
    Geo g;
    memset(&g, 0, sizeof(g));
    g.dtype = dtype;
    return linear(g, a, st);
}

}  // namespace nmm

using namespace nmm;

extern "C" {

int nmm_abi_version(void) { return NMM_ABI_VERSION; }
const char *nmm_last_error(void) { return last_error_ref().c_str(); }
uint64_t nmm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
int nmm_device_check(void) { return device_check(); }
int nmm_validate(const nmm_shape *s) { return validate(s); }

int nmm_set_option(int32_t option, int64_t value) {
    if (option < 0 || option >= NMM_OPT_COUNT) return fail(NMM_ERR_BAD_ARG, "unknown option %d", option);
    std::call_once(g_opts_once, init_opts);
    g_opts[option].store(value, std::memory_order_relaxed);
    return NMM_OK;
}
int64_t nmm_get_option(int32_t option) { return opt(option); }

int nmm_profile_begin(void) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    for (auto &r : g_prof.rec) g_prof.pool.emplace_back(r.start, r.stop);
    g_prof.rec.clear();
    g_prof.enabled = true;
    return NMM_OK;
}

int nmm_profile_end(nmm_kernel_profile *out, int32_t max_kernels) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.enabled = false;
    if (!out || max_kernels < K_COUNT) return fail(NMM_ERR_BAD_ARG, "nmm_profile_end needs room for %d kernels", (int)K_COUNT);
    static const char *names[K_COUNT] = {"gn_stats", "gn_tokens", "layernorm_pe", "temporal_attention", "linear_fp32_fma",
                                         "linear_bf16_tcgen05", "pack_params", "fused_module_tcgen05", "spatial_attention"};
    for (int k = 0; k < max_kernels; k++) { out[k].name = k < K_COUNT ? names[k] : "unused"; out[k].launches = 0; out[k].total_ms = 0; out[k].flops = 0; out[k].bytes = 0; }
    int rc = NMM_OK;
    for (auto &r : g_prof.rec) {
        float ms = 0.f;
        cudaError_t e = cudaEventSynchronize(r.stop);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.start, r.stop);
        if (e != cudaSuccess) { rc = fail(NMM_ERR_CUDA, "profile event: %s", cudaGetErrorString(e)); cudaGetLastError(); continue; }
        out[r.kid].launches += 1; out[r.kid].total_ms += ms; out[r.kid].flops += r.flops; out[r.kid].bytes += r.bytes;
        g_prof.pool.emplace_back(r.start, r.stop);
    }
    g_prof.rec.clear();
    return rc;
}

int nmm_packed_params_bytes(const nmm_shape *s, size_t *out_bytes) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!out_bytes) return fail(NMM_ERR_BAD_ARG, "out_bytes is NULL");
    *out_bytes = packed_layout(geo_of(s)).total;
    return NMM_OK;
}

int nmm_workspace_bytes(const nmm_shape *s, size_t *out_bytes) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!out_bytes) return fail(NMM_ERR_BAD_ARG, "out_bytes is NULL");
    *out_bytes = work_layout(geo_of(s)).total;
    return NMM_OK;
}

int nmm_pack_params(const nmm_shape *s, const nmm_params *src, void *packed, size_t packed_bytes, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!src || !packed) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if (src->dtype != NMM_F32 && src->dtype != NMM_BF16) return fail(NMM_ERR_BAD_ARG, "unknown source parameter dtype %d", src->dtype);
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    const PackedLayout L = packed_layout(g);
    if (packed_bytes < L.total) return fail(NMM_ERR_WORKSPACE, "packed buffer too small: %zu < %zu", packed_bytes, L.total);
    if (!aligned(packed, 256)) return fail(NMM_ERR_BAD_ARG, "packed buffer must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char *base = (char *)packed;
    const int sd = src->dtype, wd = g.dtype;
    const int64_t C = g.C;
#define PACK(srcp, off, dd, rows, cols, half)                                                        \
    do {                                                                                             \
        rc = launch_convert_rows((srcp), sd, base + (off), (dd), (rows), (cols), (half), st);        \
        if (rc != NMM_OK) return rc;                                                                 \
    } while (0)
    {
        PackedHeader hd;
        memset(&hd, 0, sizeof(hd));
        hd.magic = PACKED_MAGIC; hd.abi = NMM_ABI_VERSION; hd.dtype = g.dtype; hd.ln_fold = g.ln_fold ? 1 : 0; hd.C = g.C; hd.heads = g.heads;
        hd.layers = g.layers; hd.A = g.A; hd.max_len = g.max_len; hd.pos_enc = g.pos_enc ? 1 : 0; hd.total = L.total;
        launch_pdl(write_header_kernel, 1, 32, 0, st, hd, (PackedHeader *)(base + L.header));
        NMM_LAUNCHED("write_header_kernel");
    }
    PACK(src->gn_w, L.gn_w, NMM_F32, C, 1, 0); PACK(src->gn_b, L.gn_b, NMM_F32, C, 1, 0);
    PACK(src->proj_in_w, L.w_in, wd, C, C, 0); PACK(src->proj_in_b, L.b_in, NMM_F32, C, 1, 0);
    for (int l = 0; l < g.layers; l++) {
        const nmm_layer_params &lp = src->layer[l];
        const LayerOff &lo = L.layer[l];
        for (int i = 0; i < g.A; i++) {
            const nmm_attn_params &ap = lp.attn[i];
            const AttnOff &ao = lo.attn[i];
            PACK(ap.norm_w, ao.ln_w, NMM_F32, C, 1, 0); PACK(ap.norm_b, ao.ln_b, NMM_F32, C, 1, 0);
            const size_t wbytes = (size_t)C * C * operand_size(wd);
            PACK(ap.to_out_w, ao.wo, wd, C, C, 0); PACK(ap.to_out_b, ao.bo, NMM_F32, C, 1, 0);
            if (g.pos_enc) {
                if (ap.pe) PACK(ap.pe, ao.pe, NMM_F32, (int64_t)g.max_len, C, 0);
                else {
                    const int n = g.max_len * g.C;
                    launch_pdl(make_pe_kernel, (n + 255) / 256, 256, 0, st, (float *)(base + ao.pe), g.max_len, g.C);
                    NMM_LAUNCHED("make_pe_kernel");
                }
            }
            if (g.ln_fold) {
                // gamma-folded q|k|v weights + tables; pe.W^T needs the module's pe in the SOURCE dtype: use the caller's buffer
                // when given, else the fp32 table just generated (source dtype fp32 only)
                const void *pe_src = ap.pe;
                if (g.pos_enc && !pe_src && sd != NMM_F32) return fail(NMM_ERR_BAD_ARG, "LayerNorm folding needs the pos_encoder.pe buffer for bf16 parameters");
                if (g.pos_enc && !pe_src) pe_src = base + ao.pe;
                const void *srcs[3] = {ap.to_q, ap.to_k, ap.to_v};
                for (int m = 0; m < 3; m++) {
                    rc = fold_linear(sd, srcs[m], ap.norm_w, ap.norm_b, nullptr, g.pos_enc ? pe_src : nullptr, base + ao.wqkv + m * wbytes,
                                     (float *)(base + ao.g_qkv) + m * C, (float *)(base + ao.c_qkv) + m * C,
                                     g.pos_enc ? (float *)(base + ao.pew) + m * C : nullptr, C, C, 0, g.max_len, 3 * C, st);
                    if (rc != NMM_OK) return rc;
                }
            } else {
                PACK(ap.to_q, ao.wqkv, wd, C, C, 0); PACK(ap.to_k, ao.wqkv + wbytes, wd, C, C, 0); PACK(ap.to_v, ao.wqkv + 2 * wbytes, wd, C, C, 0);
                if (attn_fuse_weights(g) && (rc = launch_qkv_tile_order(base + ao.wqkv, base + ao.wqkv_t, (int)C, st)) != NMM_OK) return rc;
            }
            if (fused_module_weights(g)) {
                launch_pdl(wo_tail_kernel, 40, 256, 0, st, (const bf16 *)(base + ao.wo), (bf16 *)(base + ao.wo_tail), (int)C);
                NMM_LAUNCHED("wo_tail_kernel");
            }
        }
        PACK(lp.ff_norm_w, lo.ff_ln_w, NMM_F32, C, 1, 0); PACK(lp.ff_norm_b, lo.ff_ln_b, NMM_F32, C, 1, 0);
        PACK(lp.ff_proj_b, lo.b1, NMM_F32, 8 * C, 1, (int)(4 * C));
        if (g.ln_fold) {
            rc = fold_linear(sd, lp.ff_proj_w, lp.ff_norm_w, lp.ff_norm_b, lp.ff_proj_b, nullptr, base + lo.w1, (float *)(base + lo.g1),
                             (float *)(base + lo.c1), nullptr, 8 * C, C, (int)(4 * C), 0, 0, st);
            if (rc != NMM_OK) return rc;
        } else {
            PACK(lp.ff_proj_w, lo.w1, wd, 8 * C, C, (int)(4 * C));
        }
        PACK(lp.ff_out_w, lo.w2, wd, C, 4 * C, 0); PACK(lp.ff_out_b, lo.b2, NMM_F32, C, 1, 0);
    }
    PACK(src->proj_out_w, L.w_out, wd, C, C, 0); PACK(src->proj_out_b, L.b_out, NMM_F32, C, 1, 0);
#undef PACK
    if (fused_module_weights(g)) {
        // proj_in with the GroupNorm affine folded in:  (xhat * gamma + beta) . W^T + b  =  xhat . (gamma (.) W)^T + (b + beta . W^T)
        rc = fold_linear(sd, src->proj_in_w, src->gn_w, src->gn_b, src->proj_in_b, nullptr, base + L.w_in_g, (float *)(base + L.fold_tmp),
                         (float *)(base + L.b_in_g), nullptr, C, C, 0, 0, 0, st);
        if (rc != NMM_OK) return rc;
        const LayerOff &lo = L.layer[0];
        BiasList bl;
        bl.n = g.A + 2;
        bl.b[0] = (const float *)(base + L.b_in_g);
        for (int i = 0; i < g.A; i++) bl.b[1 + i] = (const float *)(base + lo.attn[i].bo);
        bl.b[g.A + 1] = (const float *)(base + lo.b2);
        float *cb = (float *)(base + L.cbias);
        launch_pdl(cumulative_bias_kernel, (unsigned)ceil_div(C, 128), 128, 0, st, cb, bl, (int)C);
        NMM_LAUNCHED("cumulative_bias_kernel");
        auto F32p = [&](size_t o) { return (const float *)(base + o); };
        for (int i = 0; i < g.A; i++) {     // cb_i | gamma_i | beta_i + pe_i[f]
            launch_pdl(vector_block_kernel, 16, 256, 0, st, (float *)(base + L.vec_attn[i]), (const float *)(cb + (size_t)i * C), F32p(lo.attn[i].ln_w),
                       F32p(lo.attn[i].ln_b), g.pos_enc ? F32p(lo.attn[i].pe) : (const float *)nullptr, g.pos_enc ? g.max_len : 1, (int)C);
            NMM_LAUNCHED("vector_block_kernel");
        }
        launch_pdl(vector_block_kernel, 16, 256, 0, st, (float *)(base + L.vec_ff), (const float *)(cb + (size_t)g.A * C), F32p(lo.ff_ln_w), F32p(lo.ff_ln_b),
                   (const float *)nullptr, 1, (int)C);
        NMM_LAUNCHED("vector_block_kernel");
        launch_pdl(vector_block_kernel, 16, 256, 0, st, (float *)(base + L.vec_fin), (const float *)(cb + (size_t)(g.A + 1) * C), F32p(L.b_out),
                   (const float *)nullptr, (const float *)nullptr, 0, (int)C);
        NMM_LAUNCHED("vector_block_kernel");
    }
    return NMM_OK;
}

static int forward_impl(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace, size_t workspace_bytes,
                        void *stream, float *stage_dump, int stage_id, const double *x_sums = nullptr, double *y_sums = nullptr);

int nmm_forward(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace, size_t workspace_bytes,
                void *stream) {
    return forward_impl(s, x, y, packed, packed_bytes, workspace, workspace_bytes, stream, nullptr, -1);
}

int nmm_forward_stats(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace, size_t workspace_bytes,
                      const double *x_sums, double *y_sums, void *stream) {
    if (x_sums != nullptr && !aligned(x_sums, 16)) return fail(NMM_ERR_BAD_ARG, "x_sums must be 16-byte aligned");
    if (y_sums != nullptr && !aligned(y_sums, 16)) return fail(NMM_ERR_BAD_ARG, "y_sums must be 16-byte aligned");
    return forward_impl(s, x, y, packed, packed_bytes, workspace, workspace_bytes, stream, nullptr, -1, x_sums, y_sums);
}

int nmm_forward_stage(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace, size_t workspace_bytes,
                      int32_t stage_id, float *stage_out, void *stream) {
    if (!stage_out || stage_id < 0) return fail(NMM_ERR_BAD_ARG, "nmm_forward_stage needs a stage id and an output buffer");
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    const Geo g = geo_of(s);
    if (!fused_module_eligible(g, s, x)) return fail(NMM_ERR_UNSUPPORTED, "nmm_forward_stage: this call does not run on the fused module kernel");
    if (stage_id > g.A + 1) return fail(NMM_ERR_BAD_ARG, "stage id %d outside [0, %d]", stage_id, g.A + 1);
    return forward_impl(s, x, y, packed, packed_bytes, workspace, workspace_bytes, stream, stage_out, stage_id);
}

// The header nmm_pack_params writes for this geometry (reading the device copy back would need a synchronisation inside nmm_forward,
// which must stay graph-capturable: nmm_forward checks packed_bytes, hosts / tests compare headers).
int nmm_packed_header(const nmm_shape *s, void *out, size_t out_bytes) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!out || out_bytes < sizeof(PackedHeader)) return fail(NMM_ERR_BAD_ARG, "nmm_packed_header needs %zu bytes", sizeof(PackedHeader));
    const Geo g = geo_of(s);
    PackedHeader hd;
    memset(&hd, 0, sizeof(hd));
    hd.magic = PACKED_MAGIC; hd.abi = NMM_ABI_VERSION; hd.dtype = g.dtype; hd.ln_fold = g.ln_fold ? 1 : 0; hd.C = g.C; hd.heads = g.heads;
    hd.layers = g.layers; hd.A = g.A; hd.max_len = g.max_len; hd.pos_enc = g.pos_enc ? 1 : 0; hd.total = packed_layout(g).total;
    memcpy(out, &hd, sizeof(hd));
    return NMM_OK;
}

static int forward_impl(const nmm_shape *s, const void *x, void *y, const void *packed, size_t packed_bytes, void *workspace, size_t workspace_bytes,
                        void *stream, float *stage_dump, int stage_id, const double *x_sums, double *y_sums) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !y || !packed || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if (x == y) return fail(NMM_ERR_BAD_ARG, "x and y must not alias");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    const PackedLayout L = packed_layout(g);
    const WorkLayout w = work_layout(g);
    if (packed_bytes != L.total)
        return fail(NMM_ERR_WORKSPACE, "packed parameter buffer of %zu bytes does not match this call's layout (%zu bytes): packed for another dtype / ln_fold / geometry?",
                    packed_bytes, L.total);
    if (workspace_bytes < w.total) return fail(NMM_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, w.total);
    if (!aligned(workspace, 1024) || !aligned(packed, 256)) return fail(NMM_ERR_BAD_ARG, "workspace must be 1024-byte and packed params 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const char *pk = (const char *)packed;
    char *ws = (char *)workspace;
    double *gn_partial = (double *)(ws + w.gn_partial);
    void *tok = ws + w.tok, *big = ws + w.big, *ctx = ws + w.ctx;
    float *h = (float *)(ws + w.h);
    auto F32 = [&](size_t off) { return (const float *)(pk + off); };

    // GroupNorm statistics over the whole tensor                                       motion_module.py:142
    // (N1: a producer that already knows the per-(b, f, group) sums of x hands them over and the pass over x is skipped)
    const double *gn_stats = gn_partial;
    int gn_nsplit = gn_splits_of(g);
    if (x_sums != nullptr) { gn_stats = x_sums; gn_nsplit = 1; }
    else if ((rc = launch_gn_stats(g, s, x, gn_partial, st)) != NMM_OK) return rc;
    float2 *stat_part = (float2 *)(ws + w.stat_part);
    // statistics of y for the next GroupNorm when the last kernel cannot emit them (fp32 modes, ragged / unaligned y, chunked runs):
    // one more pass over y with the statistics kernel, then the same [B*F*32][2] format
    auto y_sums_by_pass = [&]() -> int {
        nmm_shape sy = *s;
        sy.x_stride_b = s->y_stride_b; sy.x_stride_c = s->y_stride_c; sy.x_stride_f = s->y_stride_f;
        int r = launch_gn_stats(g, &sy, y, gn_partial, st);
        if (r != NMM_OK) return r;
        return launch_gn_partial_to_sums(g, gn_partial, y_sums, st);
    };

    // C = 320, 8 heads, 8 / 16 frames, bf16: everything else of the call is ONE kernel (fused_module.cu)
    if (fused_module_eligible(g, s, x)) {
        FusedArgs fa;
        memset(&fa, 0, sizeof(fa));
        fa.x = x; fa.y = y;
        fa.xsb = s->x_stride_b; fa.xsc = s->x_stride_c; fa.xsf = s->x_stride_f; fa.ysb = s->y_stride_b; fa.ysc = s->y_stride_c; fa.ysf = s->y_stride_f;
        fa.B = g.B; fa.F = g.F; fa.P = g.P; fa.A = g.A; fa.pos_enc = g.pos_enc ? 1 : 0;
        fa.gn_partial = gn_stats; fa.gn_splits = gn_nsplit; fa.gn_count = (double)(g.C / NMM_GN_GROUPS) * g.P; fa.gn_eps = s->eps_gn;
        const LayerOff &lo = L.layer[0];
        fa.w_in_g = pk + L.w_in_g; fa.w_out = pk + L.w_out; fa.w1 = pk + lo.w1; fa.w2 = pk + lo.w2;
        for (int i = 0; i < g.A; i++) {
            const AttnOff &ao = lo.attn[i];
            fa.wqkv_t[i] = pk + ao.wqkv_t; fa.wo[i] = pk + ao.wo; fa.wo_tail[i] = pk + ao.wo_tail;
            fa.vec_attn[i] = F32(L.vec_attn[i]);
        }
        fa.vec_ff = F32(L.vec_ff); fa.vec_fin = F32(L.vec_fin); fa.b1 = F32(lo.b1);
        fa.ln_eps = s->eps_ln;
        fa.stage_dump = stage_dump; fa.stage_id = stage_id;
        // y sums: emitted from the kernel's y store (option), or -- default, measured faster on B200: the y phase of the kernel is not
        // overlapped with tensor work, +2.2 us per tile, against ~10 us for a pass over the L2-resident y -- by a statistics pass
        const bool emit = y_sums != nullptr && opt(NMM_OPT_FUSED_Y_STATS) != 0;
        fa.y_part = emit ? stat_part : nullptr;
        if ((rc = launch_fused_module(fa, st)) != NMM_OK) return rc;
        if (emit) return launch_y_sums_tiles(stat_part, y_sums, g.B, g.F, g.P / (128 / g.F), st);
        return y_sums != nullptr ? y_sums_by_pass() : NMM_OK;
    }

    const int pc = chunk_positions(g);
    const size_t es = dtype_size(g.dtype);
    for (int p0 = 0; p0 < g.P; p0 += pc) {
        // geometry of this chunk: positions [p0, p0 + pn) of every (b, f) image; x / y offset to the chunk's first position
        const int pn = (g.P - p0 < pc) ? g.P - p0 : pc;
        Geo gc = g;
        gc.H = 1; gc.W = pn; gc.P = pn; gc.N = (int64_t)g.B * g.F * pn;
        nmm_shape sc = *s;
        sc.height = 1; sc.width = pn;
        const char *xc = (const char *)x + (size_t)p0 * es;
        char *yc = (char *)y + (size_t)p0 * es;

        // normalise + re-layout to token-major                                          :142-144
        // bf16, whole image, 64-position aligned: proj_in TMA-loads x itself and normalises the tile in shared memory (no token buffer)
        const bool gn_fused = g.dtype == NMM_BF16 && !g.ln_fold && pn == g.P && linear_tc_gn_fusable(gc.N, pn, x, s->x_stride_b, s->x_stride_c, s->x_stride_f);
        if (!gn_fused && (rc = launch_gn_tokens(gc, &sc, g, xc, gn_stats, F32(L.gn_w), F32(L.gn_b), tok, st, x_sums ? 1 : 0)) != NMM_OK) return rc;

        LinearArgs a;
        memset(&a, 0, sizeof(a));
        a.M = gc.N; a.F = g.F; a.P = pn;
        a.xsb = s->x_stride_b; a.xsc = s->x_stride_c; a.xsf = s->x_stride_f;
        a.ysb = s->y_stride_b; a.ysc = s->y_stride_c; a.ysf = s->y_stride_f;

        // LayerNorm folding (bf16 mode): every GEMM that writes the residual stream also writes a bf16 copy of it (tok2) and per-row
        // partial statistics; QKV / GEGLU then run on tok2 with gamma-folded weights and finish the normalisation in their epilogue.
        const bool fold = g.ln_fold;
        void *tok2 = ws + w.tok2;
        float *ln_part = (float *)(ws + w.ln_part);
        int nparts = 0;                                   // partial slots the last residual-writing GEMM filled
        auto producer = [&](LinearArgs &la) {            // la writes h: add the fold outputs
            if (!fold) return;
            int bn = 0, cl = 0;
            plan_linear_tc(la.M, la.N, la.K, la.epilogue, &bn, &cl);
            nparts = 2 * (la.N / bn);
            la.out = tok2; la.ln_part_out = ln_part;
        };
        auto consumer = [&](LinearArgs &la, const float *gg, const float *cc, const float *pew) {
            la.A = tok2; la.bias = nullptr; la.ln_part_in = ln_part; la.ln_nparts = nparts; la.ln_g = gg; la.ln_c = cc; la.ln_pew = pew;
            la.ln_eps = s->eps_ln;
        };
        auto clear_fold = [&](LinearArgs &la) { la.ln_part_out = nullptr; la.ln_part_in = nullptr; la.ln_pew = nullptr; la.no_h_store = 0; };

        // proj_in -> fp32 residual stream h                                             :145
        a.epilogue = NMM_EPI_STORE; a.N = g.C; a.K = g.C; a.A = tok; a.W = pk + L.w_in; a.bias = F32(L.b_in); a.h = h; a.out = nullptr;
        producer(a);
        if (gn_fused) {
            a.A = nullptr; a.gn_x = x; a.gn_partial = gn_stats; a.gn_splits = gn_nsplit;
            a.gn_count = (double)(g.C / NMM_GN_GROUPS) * g.P; a.gn_eps = s->eps_gn; a.gn_w = F32(L.gn_w); a.gn_b = F32(L.gn_b); a.gn_B = g.B;
        }
        if ((rc = linear(g, a, st)) != NMM_OK) return rc;
        a.gn_x = nullptr;
        clear_fold(a);

        for (int l = 0; l < g.layers; l++) {
            const LayerOff &lo = L.layer[l];
            for (int i = 0; i < g.A; i++) {
                const AttnOff &ao = lo.attn[i];
                // q|k|v = (LayerNorm(h) + pe[f]) . Wqkv^T                               :212, :277-278, :289,297,298
                a.epilogue = NMM_EPI_STORE; a.N = 3 * g.C; a.K = g.C; a.A = tok; a.W = pk + ao.wqkv; a.bias = nullptr; a.h = nullptr; a.out = big;
                if (fold) consumer(a, F32(ao.g_qkv), F32(ao.c_qkv), g.pos_enc ? F32(ao.pew) : nullptr);
                else if ((rc = launch_layernorm_pe(gc, &sc, h, F32(ao.ln_w), F32(ao.ln_b), g.pos_enc ? F32(ao.pe) : nullptr, tok, st)) != NMM_OK) return rc;
                // bf16, d_h 40 / 80, 8 or 16 frames: the attention runs inside the projection's epilogue (q | k | v never leave the SM)
                const bool attn_fused = attn_fuse_weights(g) && pn == g.P && linear_tc_attn_fusable(g.C, g.heads, g.F, g.P);
                if (attn_fused) {
                    a.epilogue = NMM_EPI_QKV_ATTN; a.W = pk + ao.wqkv_t; a.out = ctx; a.attn_B = g.B; a.attn_heads = g.heads;
                }
                if (planes_of(g.dtype) > 1) { a.h = (float *)big; a.out = nullptr; }      // q|k|v stay fp32 for the fp32 attention kernel
                if ((rc = linear(g, a, st)) != NMM_OK) return rc;
                clear_fold(a);
                // softmax(q k^T / sqrt(dh)) v over frames                               motion_module_new.py:258-287
                if (!attn_fused && (rc = launch_temporal_attention(gc, big, ctx, st)) != NMM_OK) return rc;
                // h = ctx . Wo^T + bo + h                                               motion_module.py:321, :213-217
                a.epilogue = NMM_EPI_RESIDUAL; a.N = g.C; a.K = g.C; a.A = ctx; a.W = pk + ao.wo; a.bias = F32(ao.bo); a.h = h; a.out = nullptr;
                producer(a);
                if ((rc = linear(g, a, st)) != NMM_OK) return rc;
                clear_fold(a);
            }
            // FeedForward: LayerNorm -> GEGLU -> Linear, + h                            :219; motion_module_new.py:441-471,497-518
            a.epilogue = NMM_EPI_GEGLU; a.N = 8 * g.C; a.K = g.C; a.A = tok; a.W = pk + lo.w1; a.bias = F32(lo.b1); a.h = nullptr; a.out = big;
            if (fold) consumer(a, F32(lo.g1), F32(lo.c1), nullptr);
            else if ((rc = launch_layernorm_pe(gc, &sc, h, F32(lo.ff_ln_w), F32(lo.ff_ln_b), nullptr, tok, st)) != NMM_OK) return rc;
            if ((rc = linear(g, a, st)) != NMM_OK) return rc;
            clear_fold(a);
            const bool last = (l == g.layers - 1);
            a.epilogue = NMM_EPI_RESIDUAL; a.N = g.C; a.K = 4 * g.C; a.A = big; a.W = pk + lo.w2; a.bias = F32(lo.b2); a.h = h; a.out = nullptr;
            if (last && g.dtype != NMM_F32) { a.out = tok; a.no_h_store = 1; }   // h + ff(...) in the GEMM operand format = the A operand of proj_out (h itself is dead)
            else producer(a);
            if ((rc = linear(g, a, st)) != NMM_OK) return rc;
            clear_fold(a);
        }
        // y = proj_out(h) back in NCHW + x                                              :152-156
        a.epilogue = NMM_EPI_OUTPUT; a.N = g.C; a.K = g.C; a.A = (g.dtype != NMM_F32) ? (const void *)tok : (const void *)h;
        a.W = pk + L.w_out; a.bias = F32(L.b_out); a.h = nullptr; a.out = nullptr; a.x = xc; a.y = yc;
        // N1: proj_out's epilogue also emits the per-(32-row block, channel) sums of y (bf16 vector path, whole-image run)
        const bool emit = y_sums != nullptr && g.dtype == NMM_BF16 && pn == g.P && output_vec_ok(a);
        a.y_part = emit ? stat_part : nullptr;
        if ((rc = linear(g, a, st)) != NMM_OK) return rc;
        a.y_part = nullptr;
        if (emit) return launch_y_sums_channels(stat_part, y_sums, g.B * g.F, g.C, g.P, st);
    }
    return y_sums != nullptr ? y_sums_by_pass() : NMM_OK;
}

// ---- per-stage entry points ------------------------------------------------------------------------------
int nmm_groupnorm_stats(const nmm_shape *s, const void *x, float *mean, float *rstd, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !mean || !rstd || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    if (workspace_bytes < gn_partial_bytes(g)) return fail(NMM_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_gn_stats(g, s, x, (double *)workspace, st)) != NMM_OK) return rc;
    return launch_gn_finalize(g, s, (const double *)workspace, mean, rstd, st);
}

int nmm_groupnorm_tokens(const nmm_shape *s, const void *x, const float *gn_w, const float *gn_b, void *tokens, void *workspace,
                         size_t workspace_bytes, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !gn_w || !gn_b || !tokens || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    if (workspace_bytes < gn_partial_bytes(g)) return fail(NMM_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_gn_stats(g, s, x, (double *)workspace, st)) != NMM_OK) return rc;
    return launch_gn_tokens(g, s, g, x, (const double *)workspace, gn_w, gn_b, tokens, st);
}

int nmm_groupnorm_linear(const nmm_shape *s, const void *x, const float *gn_w, const float *gn_b, const void *W, int32_t c_out,
                         const float *bias, float *h_out, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !gn_w || !gn_b || !W || !h_out || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    if (g.dtype != NMM_BF16) return fail(NMM_ERR_UNSUPPORTED, "nmm_groupnorm_linear is bf16 only");
    if (!linear_tc_gn_fusable(g.N, g.P, x, s->x_stride_b, s->x_stride_c, s->x_stride_f))
        return fail(NMM_ERR_UNSUPPORTED, "nmm_groupnorm_linear needs H*W %% 64 == 0, N %% 128 == 0 and 16-byte aligned x / strides");
    if (workspace_bytes < gn_partial_bytes(g)) return fail(NMM_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_gn_stats(g, s, x, (double *)workspace, st)) != NMM_OK) return rc;
    LinearArgs a;
    memset(&a, 0, sizeof(a));
    a.epilogue = NMM_EPI_STORE; a.M = g.N; a.N = c_out; a.K = g.C; a.W = W; a.bias = bias; a.h = h_out;
    a.F = g.F; a.P = g.P; a.xsb = s->x_stride_b; a.xsc = s->x_stride_c; a.xsf = s->x_stride_f;
    a.gn_x = x; a.gn_partial = (const double *)workspace; a.gn_splits = gn_splits_of(g); a.gn_count = (double)(g.C / NMM_GN_GROUPS) * g.P;
    a.gn_eps = s->eps_gn; a.gn_w = gn_w; a.gn_b = gn_b; a.gn_B = g.B;
    return launch_linear_tc(a, st);
}

static size_t gn_ws_layout(const Geo &g, size_t *stats_off) {
    const size_t part = (gn_partial_bytes(g) + 255) / 256 * 256;
    if (stats_off) *stats_off = part;
    return part + (size_t)g.B * g.F * NMM_GN_GROUPS * 2 * sizeof(float);
}

int nmm_groupnorm_workspace_bytes(const nmm_shape *s, size_t *bytes) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!bytes) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    *bytes = gn_ws_layout(geo_of(s), nullptr);
    return NMM_OK;
}

static int inflated_groupnorm_impl(const nmm_shape *s, const void *x, void *y, const float *gn_w, const float *gn_b, int32_t silu, const double *x_sums,
                                   void *workspace, size_t workspace_bytes, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !y || !gn_w || !gn_b || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    size_t stats_off = 0;
    if (workspace_bytes < gn_ws_layout(g, &stats_off)) return fail(NMM_ERR_WORKSPACE, "workspace too small");
    if (!aligned(workspace, 256)) return fail(NMM_ERR_BAD_ARG, "workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = (double *)workspace;
    float *mean = (float *)((char *)workspace + stats_off), *rstd = mean + (size_t)g.B * g.F * NMM_GN_GROUPS;
    if (x_sums != nullptr) {           // statistics handed over by the producer of x: only the apply pass touches the tensor
        if ((rc = launch_gn_finalize(g, s, x_sums, mean, rstd, st, 1)) != NMM_OK) return rc;
    } else {
        if ((rc = launch_gn_stats(g, s, x, partial, st)) != NMM_OK) return rc;
        if ((rc = launch_gn_finalize(g, s, partial, mean, rstd, st)) != NMM_OK) return rc;
    }
    return launch_gn_apply(g, s, x, y, mean, rstd, gn_w, gn_b, silu ? 1 : 0, st);
}

int nmm_inflated_groupnorm(const nmm_shape *s, const void *x, void *y, const float *gn_w, const float *gn_b, int32_t silu, void *workspace,
                           size_t workspace_bytes, void *stream) {
    return inflated_groupnorm_impl(s, x, y, gn_w, gn_b, silu, nullptr, workspace, workspace_bytes, stream);
}

int nmm_inflated_groupnorm_sums(const nmm_shape *s, const void *x, void *y, const float *gn_w, const float *gn_b, int32_t silu, const double *x_sums,
                                void *workspace, size_t workspace_bytes, void *stream) {
    if (!x_sums) return fail(NMM_ERR_BAD_ARG, "x_sums is NULL");
    return inflated_groupnorm_impl(s, x, y, gn_w, gn_b, silu, x_sums, workspace, workspace_bytes, stream);
}

int nmm_groupnorm_sums(const nmm_shape *s, const void *x, double *sums, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!x || !sums || !workspace) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    if (workspace_bytes < gn_partial_bytes(g)) return fail(NMM_ERR_WORKSPACE, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_gn_stats(g, s, x, (double *)workspace, st)) != NMM_OK) return rc;
    return launch_gn_partial_to_sums(g, (const double *)workspace, sums, st);
}

int nmm_cfg_ddim_step(int32_t dtype, int64_t n, void *latents, const void *eps_uncond, const void *eps_cond, float guidance, double alpha_t,
                      double alpha_prev, void *stream) {
    if (dtype != NMM_F32 && dtype != NMM_BF16) return fail(NMM_ERR_BAD_ARG, "dtype must be NMM_F32 or NMM_BF16");
    if (n < 0 || (n > 0 && (!latents || !eps_uncond))) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    int rc = device_check();
    if (rc != NMM_OK) return rc;
    return launch_cfg_ddim(dtype, n, latents, eps_uncond, eps_cond, guidance, alpha_t, alpha_prev, (cudaStream_t)stream);
}

int nmm_layernorm_pe(const nmm_shape *s, const float *h, const float *w, const float *b, const float *pe, void *out, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!h || !w || !b || !out) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    return launch_layernorm_pe(geo_of(s), s, h, w, b, pe, out, (cudaStream_t)stream);
}

int nmm_temporal_attention(const nmm_shape *s, const void *qkv, void *ctx, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!qkv || !ctx) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    return launch_temporal_attention(geo_of(s), qkv, ctx, (cudaStream_t)stream);
}

int nmm_qkv_attention(const nmm_shape *s, const void *tokens, const void *wqkv, void *w_scratch, void *ctx, void *stream) {
    int rc = validate(s);
    if (rc != NMM_OK) return rc;
    if (!tokens || !wqkv || !w_scratch || !ctx) return fail(NMM_ERR_BAD_ARG, "NULL argument");
    if ((rc = device_check()) != NMM_OK) return rc;
    const Geo g = geo_of(s);
    if (g.dtype != NMM_BF16 || !linear_tc_attn_fusable(g.C, g.heads, g.F, g.P))
        return fail(NMM_ERR_UNSUPPORTED, "nmm_qkv_attention: bf16, d_h in {40, 80}, frames in {8, 16}, H*W %% (128 / frames) == 0 only");
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_qkv_tile_order(wqkv, w_scratch, g.C, st)) != NMM_OK) return rc;
    LinearArgs a;
    memset(&a, 0, sizeof(a));
    a.epilogue = NMM_EPI_QKV_ATTN; a.M = g.N; a.N = 3 * g.C; a.K = g.C; a.A = tokens; a.W = w_scratch; a.out = ctx;
    a.F = g.F; a.P = g.P; a.attn_B = g.B; a.attn_heads = g.heads;
    return launch_linear_tc(a, st);
}

int nmm_linear(int32_t dtype, int32_t epilogue, int64_t M, int32_t N, int32_t K, const void *A, const void *W, const float *bias,
               float *h, void *out, const nmm_shape *s, const void *x, void *y, void *stream) {
    if (dtype != NMM_F32 && dtype != NMM_BF16 && dtype != NMM_F32X3 && dtype != NMM_F32X6) return fail(NMM_ERR_BAD_ARG, "unknown dtype %d", dtype);
    if (!A || !W || M < 0 || N <= 0 || K <= 0) return fail(NMM_ERR_BAD_ARG, "bad GEMM arguments");
    int rc = device_check();
    if (rc != NMM_OK) return rc;
    LinearArgs a;
    memset(&a, 0, sizeof(a));
    a.epilogue = epilogue; a.M = M; a.N = N; a.K = K; a.A = A; a.W = W; a.bias = bias; a.h = h; a.out = out;
    switch (epilogue) {
        case NMM_EPI_STORE: if (!h && !out) return fail(NMM_ERR_BAD_ARG, "STORE epilogue needs h or out"); break;
        case NMM_EPI_RESIDUAL:
            if (!h) return fail(NMM_ERR_BAD_ARG, "RESIDUAL epilogue needs h");
            a.no_h_store = out != nullptr;      // documented contract: with `out`, h is only read
            break;
        case NMM_EPI_GEGLU: if (!out || (N & 3)) return fail(NMM_ERR_BAD_ARG, "GEGLU epilogue needs out and N %% 4 == 0 (rows packed in groups of four)"); break;
        case NMM_EPI_OUTPUT: {
            if ((rc = validate(s)) != NMM_OK) return rc;
            if (!x || !y) return fail(NMM_ERR_BAD_ARG, "OUTPUT epilogue needs x and y");
            const Geo g = geo_of(s);
            if (g.N != M || g.C != N || s->dtype != dtype) return fail(NMM_ERR_BAD_ARG, "OUTPUT epilogue: shape does not match M/N/dtype");
            a.x = x; a.y = y; a.F = g.F; a.P = g.P;
            a.xsb = s->x_stride_b; a.xsc = s->x_stride_c; a.xsf = s->x_stride_f;
            a.ysb = s->y_stride_b; a.ysc = s->y_stride_c; a.ysf = s->y_stride_f;
            break;
        }
        default: return fail(NMM_ERR_BAD_ARG, "unknown epilogue %d", epilogue);
    }
    a.planes = planes_of(dtype);      // NMM_F32X3 / X6: A / W / out are bf16 plane tensors ([rows, 2K | 3K] / [M, 2N | 3N]); x, y fp32
    return dtype == NMM_F32 ? launch_linear_simt(a, (cudaStream_t)stream) : launch_linear_tc(a, (cudaStream_t)stream);
}

}  // extern "C"

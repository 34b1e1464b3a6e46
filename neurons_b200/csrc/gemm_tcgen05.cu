// bf16 GEMM on the 5th-generation tensor cores:  D[M,N] = A[M,K] . W[N,K]^T, fp32 accumulation in TMEM,
// fused epilogues.  This is the production kernel for every nn.Linear on the motion-module path
// (motion_module.py:145,152,289,297,298,321; motion_module_new.py:466,516).
//
// Structure (persistent, warp-specialised, one CTA per SM; CG = CTAs per tile along M):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D tiles of A (128 x 64) and of this CTA's slice of W (block_n/CG x 64),
//               128-byte swizzle, into a `stages`-deep shared-memory ring; completion via mbarrier complete_tx.
//               For the residual epilogue it also L2-prefetches the tile's fp32 residual rows.
//   warp 1      MMA issuer (one thread, of the even CTA when CG == 2): tcgen05.mma.cta_group::CG.kind::f16
//               (M = 128*CG, N = block_n, K = 16) 4x per stage; tcgen05.commit releases the stage / publishes the accumulator.
//   warp 2      TMEM allocator (2 accumulator buffers of block_n fp32 columns -> the epilogue overlaps the next tile's MMAs).
//   warps 4-11  epilogue, two warps per TMEM lane quadrant alternating 32-column chunks: tcgen05.ld (lane == output row) ->
//               bias / residual / GEGLU in registers -> the lane writes its row into a swizzled shared-memory box ->
//               ONE TMA store per chunk (cp.async.bulk.tensor, rows past M clipped by the hardware).  The residual chunk
//               arrives by TMA load into the same box (double-buffered).  proj_out's NCHW store goes through a transpose buffer.
// Both operands are K-major in global memory ([rows, K] row-major), which is exactly how activations (token-major) and
// nn.Linear weights ([out, in]) are laid out, so no transposes are ever materialised.
//
// Variants compiled from the same kernel:
//   GNA (proj_in)          the A tile is TMA-loaded straight from x[b,c,f,p] (an M-major operand: MN-major SW128 descriptor) and
//                          GroupNorm-normalised in shared memory by 4 converter warps (12-15) before the MMA reads it;
//   NMM_EPI_QKV_ATTN       A rows are (position, frame) pairs (3-D tensor map, frames before positions), N tile = q | k | v of 80
//                          channels; the epilogue dumps the tile to shared memory as bf16 and runs the temporal attention there
//                          (mma.sync core shared with attention_kernel.cu) together with 8 helper warps (12-19);
//   wide (p.wide)          256 x 320 pair tile as two N = 160 MMAs per k-step into one accumulator (long-K residual GEMMs);
//   LNF                    LayerNorm folded into producer / consumer epilogues (measured slower; kept as a tested option).
//
// Tried in round 2 and removed (correct -- 235 GPU tests green -- but slower): a "LayerNorm tail", where the tile that arrives LAST on a
// 128-row block of h (per-block arrival counter after bulk-store completion + __threadfence) runs the next LayerNorm on the block from
// L2, so that no LayerNorm kernel is launched.  With only the 8 epilogue warps on a block the tail is a chain of exposed L2 latencies
// (one row per warp: +120 us per GEMM at C = 640; 4 rows in flight per warp: +65 us; LayerNorm kernel it replaces: 12.7 us), and the
// per-tile store-completion wait + device fence serialise the epilogue.  A LayerNorm needs thousands of rows in flight, not 128.
//
// Measured bounds that shaped this (profiles/, scripts/micro/tmem_bw.cu, scripts/gemm_trace.py):
//   * tcgen05.ld moves >= 245 B/clk/SM and overlaps fully with tcgen05.mma -- TMEM reads are not the limit;
//   * a 128 x 240 tile needs 46 KB of operand fill per 480 MMA-cycles; with ~2500-cycle TMA latency under load and 3 stages the
//     mainloop starves -> cta_group::2 halves the W fill per CTA (more stages in flight per byte of shared memory);
//   * an epilogue that stores from registers with per-lane addressing costs ~1100-1400 issue cycles per 32-column chunk
//     (address arithmetic + predicates + 2 warps/SMSP) -- TMA stores cut that to a few dozen instructions.
#include <cuda.h>

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>

#include "common.cuh"
#include "attention_core.cuh"
#include "epilogue.cuh"
#include "ptx.cuh"

namespace nmm {

constexpr int TC_BM = 128, TC_BK = 64;
constexpr int TC_EPI_WARPS = 8;                           // two warps per TMEM lane quadrant, alternating column chunks
constexpr int TC_THREADS = 128 + 32 * TC_EPI_WARPS;       // warps 0-3: TMA / MMA / TMEM alloc / spare; warps 4-11: epilogue
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;            // 16 KB per stage
constexpr int TC_SMEM_MAX = 226 * 1024;                   // dynamic shared memory requested at most (227 KB is the hardware cap)
constexpr int TC_BAR_BYTES = 1024;                        // barrier area (keeps the epilogue boxes 1024-byte aligned)
constexpr int TC_EPI_BUF = 8192;                          // per epilogue warp: two 4 KB boxes (32 rows x 128 B)
constexpr int TC_XPOSE_PITCH = 33;                        // proj_out transpose buffer: floats per row (conflict-free both ways)

struct TcParams {
    int64_t M;
    int N, K;
    int block_n, stages, n_tiles, tmem_cols;
    int64_t m_tiles;
    int cluster;             // CTAs per tile along M: 1 (cta_group::1) or 2 (cta_group::2 pair, each CTA stages half of W)
    int64_t cluster_tiles;   // ceil(m_tiles / cluster) * n_tiles
    int wide;                // 1: block_n = 320 computed as two N = 160 MMAs per k-step into ONE accumulator (no TMEM double buffering); CTA pairs only
    int epi_buf;             // bytes of shared memory per epilogue warp (8 KB; 12 KB when a residual epilogue also writes a bf16 copy)
    unsigned long long *trace;   // NMM_TRACE builds only: per-tile timestamps of CTA 0 (development instrumentation)
    int debug;               // NMM_GEMM_DEBUG (timing experiments only, results invalid): 1 = epilogue does nothing, 2 = no TMA loads
    int chunk_kb;            // PL 3: k-blocks per accumulator chunk (the epilogue sums the chunks in fp32 registers); otherwise unused
};
constexpr int TC_X6_CHUNK_KB = 5;      // PL 3: K = 320 per TMEM accumulator chunk
constexpr int TC_X6_MAX_BN = 128;      // PL 3: the epilogue holds 2 x 32 columns of chunk sums per thread

// GroupNorm-fused A operand (GNA instantiation): where the statistics and affine parameters live, and the x geometry
struct GnParams {
    const double *partial;   // [b*f*32][splits][2] from gn_stats
    const float *gamma, *beta;
    int splits;
    double count;
    float eps;
    int C, F, P;
};
// QKV + attention (EPI == NMM_EPI_QKV_ATTN): geometry of the fused epilogue
struct AttnParams {
    bf16 *ctx;               // [M, C] attention output
    int C, F, P, dh;
    int ppt;                 // positions per tile = 128 / F
    int tiles_per_img;       // P / ppt
    float scale_log2e;       // d_h^-1/2 * log2(e)
};
constexpr int TC_ATTN_HELPERS = 8;                       // QKV + attention: warps 12-19 share the attention phase with the epilogue warps
constexpr int TC_ATTN_WARPS = TC_EPI_WARPS + TC_ATTN_HELPERS;
constexpr int TC_ATTN_PITCH = 3 * NMM_ATTN_TILE_CH + 8;   // elements per row of the shared-memory q|k|v tile (496 bytes)
constexpr int TC_GN_WARPS = 4;                            // GNA: warps 12-15 normalise the A tile in shared memory (one 128-byte row each)
constexpr int TC_A_HALF = TC_A_BYTES / 2;                 // GNA: the A stage is two boxes of 64 channels x 64 positions

#ifdef NMM_TRACE
#define TC_DEBUG(p) ((p).debug)
#else
#define TC_DEBUG(p) 0            // the timing experiments are compiled out of the product library
#endif
#ifdef NMM_TRACE
// event slots per tile (CTA 0 only, first TRACE_TILES tiles): 0 mma:tile start, 1 mma:accumulator free, 2 mma:first stage full,
// 3 mma:all issued, 4 prod:first load issued, 5 prod:last load issued, 6 epi(w4):before tfull wait, 7 epi:accumulator ready,
// 8..11 epi(w4): chunk k done, 12 epi(w4): released, 13 epi(w8): ready, 14 epi(w8): released
constexpr int TRACE_TILES = 48, TRACE_SLOTS = 16;
#define TRACE(tile_no, slot)                                                                          \
    do {                                                                                              \
        if (p.trace != nullptr && blockIdx.x == 0 && (tile_no) < TRACE_TILES && (threadIdx.x & 31) == 0) p.trace[(tile_no) * TRACE_SLOTS + (slot)] = clock64(); \
    } while (0)
#else
#define TRACE(tile_no, slot) do { } while (0)
#endif

// ---- swizzled shared-memory boxes shared with TMA ------------------------------------------------------------------------
// fp32 box: 32 rows x 32 columns (128 B rows), CU_TENSOR_MAP_SWIZZLE_128B: 16-byte chunk j of row r lives at chunk j ^ (r & 7).
__device__ __forceinline__ uint32_t box_f32_addr(uint32_t box, int row, int chunk) { return box + row * 128 + ((chunk ^ (row & 7)) << 4); }
// bf16 box: 32 rows x 32 columns (64 B rows), CU_TENSOR_MAP_SWIZZLE_64B: chunk j of row r lives at chunk j ^ ((r >> 1) & 3).
__device__ __forceinline__ uint32_t box_bf16_addr(uint32_t box, int row, int chunk) { return box + row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// Attention phase of the fused QKV kernel: the (position, head) problems of the shared q|k|v tile at `xb`, shared by `nw` warps (the
// 8 epilogue warps + 8 helper warps: two warps per scheduler leave the mma.sync / ldmatrix / shuffle chains latency-bound).  Two
// problems at a time per warp when the tile has enough of them; each finished problem's F x d_h block of context is copied to
// global memory by the same warp (16-byte stores; 4-byte stores straight from the accumulator fragments measured 15 % slower), so no
// block-wide barrier is needed between the math and the copy.
__device__ __forceinline__ void fused_attention_phase(const AttnParams &at, uint32_t xb, int64_t m_blk, int n_blk, int widx, int nw, int lane) {
    const int img = (int)(m_blk / at.tiles_per_img);
    const int p0 = (int)(m_blk - (int64_t)img * at.tiles_per_img) * at.ppt;
    bf16 *dst0 = at.ctx + ((int64_t)img * at.F * at.P + p0) * at.C + n_blk * NMM_ATTN_TILE_CH;
    auto run = [&](auto FF, auto DD) {
        constexpr int F_ = decltype(FF)::value, D_ = decltype(DD)::value;
        constexpr int HB_ = NMM_ATTN_TILE_CH / D_;                        // heads per tile: 2 (d_h 40) or 1 (d_h 80)
        const int nprob = at.ppt * HB_;
        auto qaddr = [&](int prob) {
            const int pl = prob / HB_, hd = prob - pl * HB_;
            return xb + (uint32_t)(pl * F_) * (TC_ATTN_PITCH * 2) + (uint32_t)(hd * D_ * 2);
        };
        auto copy_out = [&](int prob) {                                   // F rows x (d_h / 8) 16-byte chunks, all bounds compile-time
            constexpr int CPR = D_ / 8;
            const int pl = prob / HB_, hd = prob - pl * HB_;
            const uint32_t src = xb + (uint32_t)(pl * F_) * (TC_ATTN_PITCH * 2) + (uint32_t)(hd * D_ * 2);
            bf16 *dst = dst0 + (int64_t)pl * at.C + hd * D_;
#pragma unroll
            for (int i0 = 0; i0 < F_ * CPR; i0 += 32) {
                const int i = i0 + lane;
                if (i < F_ * CPR) {
                    const int f = i / CPR, v = i - f * CPR;
                    const float4 val = lds128(src + (uint32_t)f * (TC_ATTN_PITCH * 2) + (uint32_t)(v * 16));
                    *reinterpret_cast<float4 *>(dst + (int64_t)f * at.P * at.C + v * 8) = val;
                }
            }
        };
        int prob = widx;
        for (; prob + nw < nprob; prob += 2 * nw) {
            const uint32_t qb2[2] = {qaddr(prob), qaddr(prob + nw)};
            attention_problems<F_, D_, NMM_ATTN_TILE_CH, 2>(qb2, lane, at.scale_log2e, SmemQSlotStore<NMM_ATTN_TILE_CH>{qb2});
            __syncwarp();
            copy_out(prob); copy_out(prob + nw);
        }
        if (prob < nprob) {
            const uint32_t qb1[1] = {qaddr(prob)};
            attention_problems<F_, D_, NMM_ATTN_TILE_CH, 1>(qb1, lane, at.scale_log2e, SmemQSlotStore<NMM_ATTN_TILE_CH>{qb1});
            __syncwarp();
            copy_out(prob);
        }
    };
    if (at.F == 8) {
        if (at.dh == 40) run(std::integral_constant<int, 8>{}, std::integral_constant<int, 40>{});
        else run(std::integral_constant<int, 8>{}, std::integral_constant<int, 80>{});
    } else {
        if (at.dh == 40) run(std::integral_constant<int, 16>{}, std::integral_constant<int, 40>{});
        else run(std::integral_constant<int, 16>{}, std::integral_constant<int, 80>{});
    }
}

// LNF: LayerNorm-folding roles compiled in (consumer transform / producer statistics).  Kept out of the default instantiation:
// a run-time branch inside the unrolled epilogue loops costs the GEGLU epilogue its instruction-level parallelism (measured
// 128 -> 204 us at C = 320).
// PL: bf16 planes per operand.  1 = plain bf16.
// PL = 2, fp32-grade mode (NMM_F32X3).  Both operands arrive as bf16 [rows, 2K] = [hi | lo] planes (v = hi + lo + O(2^-17 v)); the K loop runs
// 3 * K / 64 k-blocks: hi.hi, hi.lo and lo.hi products accumulated in fp32 (the lo.lo term, 2^-16 relative, is dropped) -- the same
// mainloop, three passes over the planes.  GEMM-operand outputs (`out`) are written as hi | lo planes too; x / y of the OUTPUT epilogue are fp32.
// PL = 3, fp32-exact mode (NMM_F32X6).  Operands are bf16 [rows, 3K] = [hi | mid | lo] planes (v = hi + mid + lo + O(2^-24 v)); the K loop
// runs 6 * K / 64 k-blocks, one pass per product of weight >= 2^-16, SMALL TERMS FIRST: lo.hi, mid.mid, hi.lo (2^-16), mid.hi, hi.mid (2^-8),
// hi.hi (the dropped mid.lo, lo.mid, lo.lo are <= 2^-24).  The tensor core's fp32 accumulation is not round-to-nearest: measured on a B200,
// one accumulator over the whole k-block sequence gave an error that grows about linearly with K (3.8e-5 at K = 5120 on N(0, 1) outputs,
// 2.4x the FMA GEMM's).  So the sequence runs in chunks of p.chunk_kb k-blocks (K = 320), each into a fresh accumulator of the two TMEM
// buffers; the epilogue warps add the chunk results in fp32 registers (round to nearest) while the next chunk accumulates, write the sum back
// into the last chunk's accumulator and drain that as usual.  Small terms first keeps the small passes' roundings at their own magnitude
// (tests/test_fp32_exact_tc.py emulates both orders).  `out` is written as hi | mid | lo planes; fp32 outputs stay fp32.
template <int EPI, int CG, bool LNF, bool GNA, int PL>
__global__ void __launch_bounds__(EPI == NMM_EPI_QKV_ATTN ? TC_THREADS + 32 * TC_ATTN_HELPERS : GNA ? TC_THREADS + 32 * TC_GN_WARPS : TC_THREADS, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w,
                 const __grid_constant__ CUtensorMap tm_h,      // fp32 [M,N], box 32 x 32, 128-byte swizzle (residual load / h store)
                 const __grid_constant__ CUtensorMap tm_o,      // bf16 [M,N or N/2], box 32 x 32, 64-byte swizzle (`out` store)
                 TcParams p, EpiParams e, GnParams gn, AttnParams at) {
    // CG == 1: one CTA per 128 x block_n tile (tcgen05.mma.cta_group::1).
    // CG == 2: a CTA pair (cluster of 2 along M) computes a 256 x block_n tile with ONE tcgen05.mma.cta_group::2 stream issued
    //          by the even CTA: each CTA stages its own 128 rows of A and HALF of the W tile (block_n/2 rows); the tensor core
    //          reads the two W halves from both CTAs' shared memory and each CTA's TMEM receives its own 128 x block_n accumulator.
    extern __shared__ unsigned char smem_raw[];
    const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;     // SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t b_rows = (uint32_t)p.block_n / CG;                           // W rows staged by this CTA
    const uint32_t stage_bytes = TC_A_BYTES + b_rows * TC_BK * 2;
    const uint32_t bar_base = smem_base + (uint32_t)p.stages * stage_bytes;
    // barrier area: full[stages], empty[stages], tmem_full[2], tmem_empty[2], TMEM base address; +512: per-epilogue-warp load barriers
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (p.stages + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * p.stages + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * p.stages + 2 + s); };
    const uint32_t tmem_slot = bar_base + 8u * (2 * p.stages + 4);
    auto load_bar = [&](int ew, int b) { return bar_base + 512u + 8u * (ew * 2 + b); };
    auto conv_bar = [&](int s) { return bar_base + 768u + 8u * s; };          // GNA: A tile of stage s normalised
    const uint32_t epi_base = bar_base + TC_BAR_BYTES;                          // 8 x 8 KB, 1024-byte aligned

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nk = (p.K + TC_BK - 1) / TC_BK;                        // k-blocks of one operand plane
    const int num_kb = PL == 3 ? 6 * nk : PL == 2 ? 3 * nk : nk;
    // PL = 2: k-block kb = pass t * nk + j multiplies A plane (t == 2 ? lo : hi) by W plane (t == 1 ? lo : hi); small terms last.
    // PL = 3: pass t multiplies A plane (0x46 >> 2t) & 3 by W plane (0x124 >> 2t) & 3 (plane 0 = hi, 1 = mid, 2 = lo): the order above.
    auto a_col = [&](int kb) {
        if constexpr (PL == 3) { const int t = kb / nk, j = kb - t * nk; return (((0x46 >> (2 * t)) & 3) * nk + j) * TC_BK; }
        else if constexpr (PL == 2) { const int t = kb / nk, j = kb - t * nk; return (t == 2 ? nk + j : j) * TC_BK; }
        else return kb * TC_BK;
    };
    auto w_col = [&](int kb) {
        if constexpr (PL == 3) { const int t = kb / nk, j = kb - t * nk; return (((0x124 >> (2 * t)) & 3) * nk + j) * TC_BK; }
        else if constexpr (PL == 2) { const int t = kb / nk, j = kb - t * nk; return (t == 1 ? nk + j : j) * TC_BK; }
        else return kb * TC_BK;
    };
    // Tile schedule: a cluster walks (m_group, n_blk) pairs; CTA `rank` of the cluster owns m-block m_group*CG + rank.
    // Both CTAs of a pair run the same number of iterations (a phantom m-block past the end is all zero-fill + clipped).
    // rank inside the (CG, 1, 1) cluster = blockIdx.x % CG, taken from blockIdx on purpose: the compiler must KNOW it is uniform.  With
    // %cluster_ctarank the leader-only MMA role compiled as divergent code -- every tcgen05.mma / TMA operand was built in vector
    // registers and moved to the uniform file by a waterfall loop, ~100 issue cycles per MMA (more than an N = 160 MMA takes to run).
    const uint32_t rank = CG > 1 ? (blockIdx.x % (unsigned)CG) : 0u;
    const bool leader = rank == 0;
    const int64_t cluster_id = blockIdx.x / CG, num_clusters = gridDim.x / CG;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a);
        ptx::prefetch_tensormap(&tm_w);
        if (EPI == NMM_EPI_RESIDUAL || e.h != nullptr) ptx::prefetch_tensormap(&tm_h);
        if (e.out != nullptr) ptx::prefetch_tensormap(&tm_o);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; s++) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
        // tmem_empty collects one arrive per epilogue warp of every CTA of the pair (it lives in the MMA-issuing CTA)
        for (int s = 0; s < 2; s++) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), TC_EPI_WARPS * CG); }
        for (int w = 0; w < TC_EPI_WARPS; w++) { ptx::mbar_init(load_bar(w, 0), 1); ptx::mbar_init(load_bar(w, 1), 1); }
        if (GNA) for (int s = 0; s < p.stages; s++) ptx::mbar_init(conv_bar(s), TC_GN_WARPS);
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc<CG>(tmem_slot, (uint32_t)p.tmem_cols);
    // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch) overlapped the previous kernel's tail.  Each role
    // executes griddepcontrol.wait itself, right before it first touches memory the previous kernel may have written -- the producer
    // only after it has put the first stages' WEIGHT tiles in flight (weights are never written by a kernel of the stream).
    pdl_launch_dependents();
    ptx::tc_fence_before();
    if (CG > 1) ptx::cluster_sync();                 // the peer's barriers must exist before any remote arrive / complete_tx
    else __syncthreads();
    ptx::tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 0) {
        // ===================== TMA producer (every CTA: its A rows, its slice of W) =====================
        // (the whole warp runs the schedule and the barrier waits; one elected lane issues -- keeps every TMA operand in uniform registers)
        {
            int stage = 0; uint32_t phase = 0;
            int tile_no = 0;
            // W tile of k-block kb -> the stage (any time: weights are constant); A tile -> the stage (after griddepcontrol.wait)
            auto issue_w = [&](int kb, int n_blk, uint32_t sa, uint32_t bar) {
                if constexpr (CG == 1) {
                    ptx::tma_load_2d(&tm_w, bar, sa + TC_A_BYTES, w_col(kb), n_blk * p.block_n);
                } else {
                    const uint32_t bar0 = bar & ptx::PEER_MASK;
                    if (p.wide) {      // two N = 160 blocks, this CTA stages its 80-row half of each
                        const uint32_t hb = b_rows / 2;
                        ptx::tma_load_2d_2sm(&tm_w, bar0, sa + TC_A_BYTES, w_col(kb), n_blk * p.block_n + (int)(rank * hb));
                        ptx::tma_load_2d_2sm(&tm_w, bar0, sa + TC_A_BYTES + hb * TC_BK * 2, w_col(kb), n_blk * p.block_n + p.block_n / 2 + (int)(rank * hb));
                    } else {
                        ptx::tma_load_2d_2sm(&tm_w, bar0, sa + TC_A_BYTES, w_col(kb), n_blk * p.block_n + (int)(rank * b_rows));
                    }
                }
            };
            auto issue_a = [&](int kb, int64_t m_blk, uint32_t sa, uint32_t bar, const int (&gp)[2], const int (&gf)[2], const int (&gb)[2]) {
                if constexpr (EPI == NMM_EPI_QKV_ATTN) {
                    // A rows = (position, frame) pairs of one image: box (64 channels, F frames, 128/F positions) of the tokens
                    // viewed as (c, b*F + f, p) -> shared-memory row pl * F + f, the attention tile order
                    const int img = (int)(m_blk / at.tiles_per_img);
                    ptx::tma_load_3d(&tm_a, bar, sa, kb * TC_BK, img * at.F, (int)(m_blk - (int64_t)img * at.tiles_per_img) * at.ppt);
                } else if constexpr (GNA) {
                    // A = x[b, kb*64 .. +64 channels, f, 64 positions] for each half of the 128-token tile (M-major boxes)
                    ptx::tma_load_4d(&tm_a, bar, sa, gp[0], kb * TC_BK, gf[0], gb[0]);
                    ptx::tma_load_4d(&tm_a, bar, sa + TC_A_HALF, gp[1], kb * TC_BK, gf[1], gb[1]);
                } else if constexpr (CG == 1) {
                    ptx::tma_load_2d(&tm_a, bar, sa, a_col(kb), (int32_t)(m_blk * TC_BM));
                } else {
                    ptx::tma_load_2d_2sm(&tm_a, bar & ptx::PEER_MASK, sa, a_col(kb), (int32_t)(m_blk * TC_BM));
                }
            };
            // both CTAs' bytes of a pair are counted on the even CTA's barrier (the only one the MMA thread waits on)
            auto expect = [&](uint32_t bar) { if (CG == 1 || leader) ptx::mbar_expect_tx(bar, (uint32_t)CG * stage_bytes); };
            // the first tile's first stages: weights before the dependency wait, activations after it
            int pre = 0;
            if (!(TC_DEBUG(p) & 2)) {
                pre = num_kb < p.stages ? num_kb : p.stages;
                if (ptx::elect_one()) {
                    const int n_blk0 = (int)(cluster_id % p.n_tiles);
                    for (int kb = 0; kb < pre; kb++) {
                        expect(full_bar(kb));
                        issue_w(kb, n_blk0, smem_base + (uint32_t)kb * stage_bytes, full_bar(kb));
                    }
                }
                __syncwarp();
            }
            pdl_wait();
            for (int64_t ct = cluster_id; ct < p.cluster_tiles; ct += num_clusters, tile_no++) {
                const int64_t m_grp = ct / p.n_tiles;
                const int n_blk = (int)(ct - m_grp * p.n_tiles);
                const int64_t m_blk = m_grp * CG + rank;
                if constexpr (EPI == NMM_EPI_RESIDUAL) {
                    // the epilogue will read-modify-write this tile's fp32 residual rows: pull them into L2 now
                    if (!(TC_DEBUG(p) & 2) && ptx::elect_one())
                        for (int c0 = 0; c0 < p.block_n; c0 += 32)
                            for (int r0 = 0; r0 < TC_BM; r0 += 32)
                                ptx::tma_prefetch_l2_2d(&tm_h, n_blk * p.block_n + c0, (int32_t)(m_blk * TC_BM + r0));
                }
                int gp[2] = {0, 0}, gf[2] = {0, 0}, gb[2] = {0, 0};     // GNA: (position, frame, batch) of the tile's two 64-token halves
                if constexpr (GNA) {
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        const int64_t n = m_blk * TC_BM + 64 * j;
                        const int bf = (int)(n / gn.P);
                        gp[j] = (int)(n - (int64_t)bf * gn.P); gb[j] = bf / gn.F; gf[j] = bf - gb[j] * gn.F;
                    }
                }
                for (int kb = 0; kb < num_kb; kb++) {
                    const bool prefilled = tile_no == 0 && kb < pre;     // W already in flight, expect_tx already posted
                    if (!prefilled) ptx::mbar_wait(empty_bar(stage), phase ^ 1u);       // the MMAs that read this stage have retired
                    if (kb == 0) TRACE(tile_no, 4);
                    if (kb == num_kb - 1) TRACE(tile_no, 5);
                    const uint32_t sa = smem_base + (uint32_t)stage * stage_bytes;
                    if (ptx::elect_one()) {
                        if (TC_DEBUG(p) & 2) {                              // timing experiment: MMA on whatever is in shared memory
                            if (leader) ptx::mbar_arrive(full_bar(stage));
                        } else {
                            if (!prefilled) expect(full_bar(stage));
                            issue_a(kb, m_blk, sa, full_bar(stage), gp, gf, gb);
                            if (!prefilled) issue_w(kb, n_blk, sa, full_bar(stage));
                        }
                    }
                    __syncwarp();
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (one thread of the even CTA) =====================
        // (whole warp; one elected lane issues the tcgen05 instructions)
        if (leader) {
            const uint32_t n_mma = p.wide ? (uint32_t)p.block_n / 2 : (uint32_t)p.block_n;      // columns per MMA instruction
            const uint32_t idesc = ptx::umma_idesc_bf16(TC_BM * CG, n_mma) | (GNA ? ptx::UMMA_IDESC_A_MN_MAJOR : 0u);
            int stage = 0; uint32_t phase = 0;
            int as = 0; uint32_t aphase = 0;
            int tile_no = 0;
            for (int64_t ct = cluster_id; ct < p.cluster_tiles; ct += num_clusters, tile_no++) {
                TRACE(tile_no, 0);
                ptx::mbar_wait(tempty_bar(as), aphase ^ 1u);           // every epilogue warp (of both CTAs) drained this accumulator
                TRACE(tile_no, 1);
                ptx::tc_fence_after();
                uint32_t d_tmem = tmem_base + (uint32_t)(as * p.block_n);
                for (int kb = 0; kb < num_kb; kb++) {
                    int kc = kb;                                              // k-block index inside the current accumulator
                    if constexpr (PL == 3) {
                        kc = kb % p.chunk_kb;
                        if (kc == 0 && kb > 0) {                              // chunk boundary: publish this accumulator, go on in the other buffer
                            if (ptx::elect_one()) ptx::umma_commit<CG>(tfull_bar(as));
                            __syncwarp();
                            if (++as == 2) { as = 0; aphase ^= 1u; }
                            ptx::mbar_wait(tempty_bar(as), aphase ^ 1u);
                            ptx::tc_fence_after();
                            d_tmem = tmem_base + (uint32_t)(as * p.block_n);
                        }
                    }
                    // TMA bytes (of both CTAs) have landed; GNA: ... and the converter warps have normalised the A tile
                    ptx::mbar_wait(GNA ? conv_bar(stage) : full_bar(stage), phase);
                    if (kb == 0) TRACE(tile_no, 2);
                    ptx::tc_fence_after();
                    const uint32_t sa = smem_base + (uint32_t)stage * stage_bytes;
                    const uint64_t b_desc = ptx::umma_smem_desc_sw128(sa + TC_A_BYTES);
                    if (ptx::elect_one()) {
                    if constexpr (GNA) {
                        // M-major A: 64-position blocks 8 KB apart (LBO), 8-channel groups 1 KB apart (SBO); K = 16 channels = 2 KB
                        const uint64_t a_desc = ptx::umma_smem_desc_mn_sw128(sa, TC_A_HALF, 1024);
                        if (TC_DEBUG(p) & 16) {            // timing experiment: K-major descriptors on the same bytes (results invalid)
                            const uint64_t a_k = ptx::umma_smem_desc_sw128(sa);
                            const uint32_t idk = idesc & ~ptx::UMMA_IDESC_A_MN_MAJOR;
#pragma unroll
                            for (int k = 0; k < TC_BK / 16; k++)
                                ptx::umma_bf16<CG>(d_tmem, a_k + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), idk, (kb | k) != 0 ? 1u : 0u);
                        } else
#pragma unroll
                        for (int k = 0; k < TC_BK / 16; k++)
                            ptx::umma_bf16<CG>(d_tmem, a_desc + (uint64_t)(k * (2048 >> 4)), b_desc + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
                    } else {
                        const uint64_t a_desc = ptx::umma_smem_desc_sw128(sa);
                        if (p.wide) {
                            // second N block: its rows follow the first block's in this CTA's W stage (n_mma / CG rows x 128 bytes further)
                            const uint64_t b_desc2 = ptx::umma_smem_desc_sw128(sa + TC_A_BYTES + (n_mma / CG) * TC_BK * 2);
#pragma unroll
                            for (int k = 0; k < TC_BK / 16; k++) {
                                ptx::umma_bf16<CG>(d_tmem, a_desc + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), idesc, (kc | k) != 0 ? 1u : 0u);
                                ptx::umma_bf16<CG>(d_tmem + n_mma, a_desc + (uint64_t)(k * 2), b_desc2 + (uint64_t)(k * 2), idesc, (kc | k) != 0 ? 1u : 0u);
                            }
                        } else {
#pragma unroll
                            for (int k = 0; k < TC_BK / 16; k++)         // +32 bytes per K=16 step inside the swizzle atom
                                ptx::umma_bf16<CG>(d_tmem, a_desc + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), idesc, (kc | k) != 0 ? 1u : 0u);
                        }
                    }
                    ptx::umma_commit<CG>(empty_bar(stage));               // stage reusable (in both CTAs) once these MMAs retire
                    }
                    __syncwarp();
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
                if (ptx::elect_one()) ptx::umma_commit<CG>(tfull_bar(as));    // accumulator complete (signalled in both CTAs)
                __syncwarp();
                TRACE(tile_no, 3);
                if (p.wide) aphase ^= 1u;                                 // single accumulator: its barriers change phase every tile
                else if (++as == 2) { as = 0; aphase ^= 1u; }
            }
        }
    } else if (EPI == NMM_EPI_QKV_ATTN && warp >= 4 + TC_EPI_WARPS) {
        // ===================== attention helpers (QKV + attention): share the tile's problems with the epilogue warps =============
        pdl_wait();
        const uint32_t xb = epi_base;
        for (int64_t ct = cluster_id; ct < p.cluster_tiles; ct += num_clusters) {
            const int64_t m_grp = ct / p.n_tiles;
            const int n_blk = (int)(ct - m_grp * p.n_tiles);
            if (TC_DEBUG(p) & 1) break;                                                  // (timing experiment without epilogue: no barriers either)
            asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_ATTN_WARPS) : "memory");     // the tile has been dumped
            fused_attention_phase(at, xb, m_grp * CG + rank, n_blk, warp - 4, TC_ATTN_WARPS, lane);
            asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_ATTN_WARPS) : "memory");     // done with the tile
        }
    } else if (GNA && warp >= 4 + TC_EPI_WARPS) {
        // ===================== GroupNorm converter (GNA): normalise the A tile in place =====================
        // Thread (j, row): the 128-byte row of channel kb*64 + row in half j (64 positions of image bf_j).  The affine is per
        // (image, channel), so the 128-byte swizzle inside the row is irrelevant; the 16-byte chunks are visited in a rotated
        // order so that 8 consecutive lanes hit 8 different bank groups.
        pdl_wait();
        const int t = (int)threadIdx.x - 32 * (4 + TC_EPI_WARPS);
        const int j = t >> 6, row = t & 63;
        const int cpg = gn.C / NMM_GN_GROUPS;
        // gamma / beta of every channel -> shared memory once per CTA (a per-k-block global load would sit on the converter's
        // critical path: ~L2 latency per 64 channels)
        float *sm_gb = reinterpret_cast<float *>(smem_raw + (epi_base + (uint32_t)TC_EPI_WARPS * (uint32_t)p.epi_buf - ptx::smem_u32(smem_raw)));
        const int kpad = num_kb * TC_BK;
        for (int c = t; c < kpad; c += 32 * TC_GN_WARPS) {
            sm_gb[c] = c < gn.C ? __ldg(gn.gamma + c) : 0.f;              // channels past C: zero rows (W's columns there are zero-filled too)
            sm_gb[kpad + c] = c < gn.C ? __ldg(gn.beta + c) : 0.f;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_GN_WARPS) : "memory");     // converter warps only
        int stage = 0; uint32_t phase = 0;
        for (int64_t ct = cluster_id; ct < p.cluster_tiles; ct += num_clusters) {
            const int64_t m_blk = (ct / p.n_tiles) * CG + rank;
            const int bf = (int)((m_blk * TC_BM + 64 * j) / gn.P);
            // lane g holds mean / rstd of group g of image bf (all 32 lanes of a warp share j, hence bf)
            float mean_g, rstd_g;
            gn_finalize_one(gn.partial, bf * NMM_GN_GROUPS + lane, gn.splits, gn.count, gn.eps, mean_g, rstd_g);
            for (int kb = 0; kb < num_kb; kb++) {
                const int c = kb * TC_BK + row;
                const int grp = min(c / cpg, NMM_GN_GROUPS - 1);
                const float mu = __shfl_sync(0xffffffffu, mean_g, grp), rs = __shfl_sync(0xffffffffu, rstd_g, grp);
                const float ca = rs * sm_gb[c], cb = sm_gb[kpad + c] - mu * ca;
                ptx::mbar_wait(full_bar(stage), phase);
                const uint32_t rbase = smem_base + (uint32_t)stage * stage_bytes + (uint32_t)(j * TC_A_HALF + row * 128);
                const uint64_t ca2 = f32x2_pack(ca, ca), cb2 = f32x2_pack(cb, cb);
                if (!(TC_DEBUG(p) & 4)) {
                    // all 8 loads first (independent, pipelined), then the arithmetic, then the stores
                    uint32_t w[8][4];
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const uint32_t addr = rbase + (uint32_t)(((i + row) & 7) << 4);
                        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[i][0]), "=r"(w[i][1]), "=r"(w[i][2]), "=r"(w[i][3]) : "r"(addr) : "memory");
                    }
#pragma unroll
                    for (int i = 0; i < 8; i++) {
#pragma unroll
                        for (int k = 0; k < 4; k++) {      // both bf16 halves of the word through one packed fp32x2 FMA (same rounding as fmaf)
                            float lo, hi;
                            f32x2_unpack(f32x2_fma(f32x2_pack(bf16_lo(w[i][k]), bf16_hi(w[i][k])), ca2, cb2), lo, hi);
                            w[i][k] = pack_bf16x2(lo, hi);
                        }
                        sts128(rbase + (uint32_t)(((i + row) & 7) << 4), w[i][0], w[i][1], w[i][2], w[i][3]);
                    }
                }
                if (!(TC_DEBUG(p) & 8)) ptx::fence_proxy_async();               // generic-proxy writes -> visible to the tensor core's async proxy
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(conv_bar(stage));
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp >= 4 && warp < 4 + TC_EPI_WARPS) {
        // ===================== epilogue (every CTA: its own 128 TMEM lanes) =====================
        pdl_wait();
        const int ew = warp - 4;
        const int q = warp & 3;                                           // TMEM lane quadrant this warp may access
        const int half = ew >> 2;                                         // which of the quadrant's two warps
        const uint32_t box0 = epi_base + (uint32_t)ew * (uint32_t)p.epi_buf, box1 = box0 + 4096u, box2 = box0 + 8192u;
        // LayerNorm folding, consumer side: per-row mean / rstd of the A rows from the producer's partial sums (lane == row)
        const bool ln_in = LNF && e.ln_part_in != nullptr;
        float *xpose = reinterpret_cast<float *>(smem_raw + (box0 - ptx::smem_u32(smem_raw)));      // proj_out transpose buffer
        uint32_t lph0 = 0u, lph1 = 0u;                                    // phases of this warp's two residual-load barriers
        int as = 0; uint32_t aphase = 0;
        int tile_no = 0;
        for (int64_t ct = cluster_id; ct < p.cluster_tiles; ct += num_clusters, tile_no++) {
            const int64_t m_grp = ct / p.n_tiles;
            const int n_blk = (int)(ct - m_grp * p.n_tiles);
            const int64_t m_blk = m_grp * CG + rank;
            const int64_t row0 = m_blk * TC_BM + q * 32;
            if constexpr (PL == 3) {
                // the chunks of this tile (see PL above): every warp adds its columns of each chunk into fp32 running sums and releases the
                // buffer; the last chunk's accumulator receives the sum and is drained below like any accumulator.  The sums (this lane's
                // row, 64 columns) live in the warp's first two epilogue boxes, 16-byte slots XOR-rotated by lane (conflict-free)
                const int nch = (num_kb + p.chunk_kb - 1) / p.chunk_kb;
                const uint32_t box0c = epi_base + (uint32_t)ew * (uint32_t)p.epi_buf;
                auto slot = [&](int v) { return box0c + (uint32_t)lane * 256u + (uint32_t)(((v ^ lane) & 15) << 4); };
                if (lane == 0) ptx::bulk_wait_read0();                    // the previous tile's stores have read the boxes
                __syncwarp();
                for (int ch = 0; ch < nch; ch++) {
                    ptx::mbar_wait(tfull_bar(as), aphase);
                    ptx::tc_fence_after();
                    const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * p.block_n);
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const int col = EPI == NMM_EPI_GEGLU ? half * 64 + 32 * i : half * 32 + 64 * i;     // the columns this warp drains below
                        if (col < p.block_n) {
                            uint32_t r[32];
                            ptx::tmem_ld32(tb + (uint32_t)col, r);
                            ptx::tmem_ld_wait();
#pragma unroll
                            for (int v = 0; v < 8; v++) {
                                if (ch > 0) {
                                    const float4 s4 = lds128(slot(8 * i + v));
                                    r[4 * v] = __float_as_uint(s4.x + __uint_as_float(r[4 * v]));
                                    r[4 * v + 1] = __float_as_uint(s4.y + __uint_as_float(r[4 * v + 1]));
                                    r[4 * v + 2] = __float_as_uint(s4.z + __uint_as_float(r[4 * v + 2]));
                                    r[4 * v + 3] = __float_as_uint(s4.w + __uint_as_float(r[4 * v + 3]));
                                }
                                if (ch < nch - 1) sts128(slot(8 * i + v), r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]);
                            }
                            if (ch == nch - 1) ptx::tmem_st32(tb + (uint32_t)col, r);
                        }
                    }
                    if (ch == nch - 1) {
                        ptx::tmem_st_wait();
                        ptx::fence_proxy_async();                         // generic writes to the boxes before TMA reuses them
                        __syncwarp();
                        break;
                    }
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (CG == 1) ptx::mbar_arrive(tempty_bar(as));
                        else ptx::mbar_arrive_cluster(tempty_bar(as) & ptx::PEER_MASK);
                    }
                    if (++as == 2) { as = 0; aphase ^= 1u; }
                }
            }
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * p.block_n);
            if (warp == 4 && lane == 0) TRACE(tile_no, 6);
            float ln_mu = 0.f, ln_rstd = 0.f;
            const float *pew_row = nullptr;
            if (ln_in) {
                const int64_t row = row0 + lane;
                if (row < p.M) {
                    float s1 = 0.f, s2 = 0.f;
                    const float2 *pp = reinterpret_cast<const float2 *>(e.ln_part_in) + row * e.ln_nparts;
                    for (int i = 0; i < e.ln_nparts; i++) { const float2 t2 = __ldg(pp + i); s1 += t2.x; s2 += t2.y; }
                    const float inv = 1.0f / (float)e.ln_K;
                    ln_mu = s1 * inv;
                    ln_rstd = rsqrtf(fmaxf(s2 * inv - ln_mu * ln_mu, 0.f) + e.ln_eps);
                    if (e.ln_pew != nullptr) pew_row = e.ln_pew + (int64_t)((row / e.P) % e.F) * e.N;
                }
            }
            float st1 = 0.f, st2 = 0.f;                                  // producer side: partial statistics of this lane's row
            bool waited = false;
            auto wait_acc = [&]() {
                if (!waited) {
                    ptx::mbar_wait(tfull_bar(as), aphase);
                    ptx::tc_fence_after();
                    waited = true;
                    if (warp == 4 && lane == 0) TRACE(tile_no, 7);
                    if (warp == 8 && lane == 0) TRACE(tile_no, 13);
                }
            };
            if (TC_DEBUG(p) & 1) {
                // timing experiment: drain nothing
            } else if constexpr (EPI == NMM_EPI_QKV_ATTN) {
                // ---- QKV + attention: the 128 x 240 accumulator tile is q | k | v (80 channels each) of 128/F positions x F frames.
                // 1. every warp dumps its 32 rows x half of the columns as bf16 into the shared q|k|v tile (row = TMEM lane =
                //    pl * F + f: consecutive lanes -> consecutive 496-byte rows, conflict-free) and releases the accumulator;
                // 2. one warp per (position, head): softmax(q k^T / sqrt d) v on mma.sync, result into the q slot (attention_core.cuh);
                // 3. the q slots (128 rows x 160 bytes) go to ctx with 16-byte stores.
                const uint32_t xb = epi_base;                           // the epilogue buffers hold the tile (63.5 KB of 64 KB)
                wait_acc();
                {
                    const uint32_t rowaddr = xb + (uint32_t)(q * 32 + lane) * (TC_ATTN_PITCH * 2);
                    // half 0: columns [0, 128) = 4 x 32; half 1: [128, 240) = 3 x 32 + 16.  Two TMEM loads in flight per wait.
                    auto put8 = [&](int c, const uint32_t *r) {          // 8 fp32 accumulator columns -> 8 bf16 = one 16-byte store
                        sts128(rowaddr + (uint32_t)(c * 2), pack_bf16x2(__uint_as_float(r[0]), __uint_as_float(r[1])), pack_bf16x2(__uint_as_float(r[2]), __uint_as_float(r[3])),
                               pack_bf16x2(__uint_as_float(r[4]), __uint_as_float(r[5])), pack_bf16x2(__uint_as_float(r[6]), __uint_as_float(r[7])));
                    };
                    const int cbeg = half ? 128 : 0;
#pragma unroll
                    for (int k = 0; k < 2; k++) {
                        const int c0 = cbeg + 64 * k;
                        uint32_t ra[32], rb[32];
                        ptx::tmem_ld32(t_row + (uint32_t)c0, ra);
                        if (k == 0 || !half) {
                            ptx::tmem_ld32(t_row + (uint32_t)(c0 + 32), rb);
                            ptx::tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 4; j++) { put8(c0 + 8 * j, ra + 8 * j); put8(c0 + 32 + 8 * j, rb + 8 * j); }
                        } else {                                             // half 1, second step: 32 + 16 columns (192 .. 239)
                            uint32_t rc[16];
                            ptx::tmem_ld16(t_row + (uint32_t)(c0 + 32), rc);
                            ptx::tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 4; j++) put8(c0 + 8 * j, ra + 8 * j);
#pragma unroll
                            for (int j = 0; j < 2; j++) put8(c0 + 32 + 8 * j, rc + 8 * j);
                        }
                    }
                }
                if (warp == 4 && lane == 0) TRACE(tile_no, 8);
                // the accumulator is drained: hand it back to the MMA warp before the attention math
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(tempty_bar(as));
                asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_ATTN_WARPS) : "memory");     // the whole q|k|v tile is in shared memory
                if (warp == 4 && lane == 0) TRACE(tile_no, 9);
                fused_attention_phase(at, xb, m_blk, n_blk, ew, TC_ATTN_WARPS, lane);
                asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_ATTN_WARPS) : "memory");     // every warp is done with the tile: free for the next dump
                if (warp == 4 && lane == 0) TRACE(tile_no, 12);
                if (++as == 2) { as = 0; aphase ^= 1u; }
                continue;
            } else if constexpr (EPI == NMM_EPI_OUTPUT) {
                // y[b,c,f,p] = acc + bias[c] + x[b,c,f,p]: the output is channel-major, rows (p) are the contiguous axis
                if (e.nchw_vec) {
                    // 32 x 32 chunk through the transpose buffer (pitch 33: conflict-free both ways); afterwards 4 lanes own
                    // 32 consecutive positions of one channel -> 16-byte loads of x and stores of y, 64 contiguous bytes per channel
                    const int cq = lane >> 2, rg = lane & 3;
                    const int64_t rowg = row0 + 8 * rg;                      // first of this lane's 8 rows
                    const bool rows_ok = row0 < p.M;                          // M % 32 == 0 on this path: all-or-nothing per warp
                    const int64_t bfi = rowg / e.P;
                    const int pp = (int)(rowg - bfi * e.P);
                    const int64_t bb = bfi / e.F, ff = bfi - bb * e.F;
                    const bf16 *xrow = reinterpret_cast<const bf16 *>(e.x) + bb * e.xsb + ff * e.xsf + pp;
                    bf16 *yrow = reinterpret_cast<bf16 *>(e.y) + bb * e.ysb + ff * e.ysf + pp;
                    for (int c0 = half * 32; c0 < p.block_n; c0 += 64) {
                        const int col0 = n_blk * p.block_n + c0;
                        uint4 xin[4];
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            xin[j] = rows_ok ? __ldg(reinterpret_cast<const uint4 *>(xrow + (int64_t)(col0 + cq + 8 * j) * e.xsc)) : make_uint4(0u, 0u, 0u, 0u);
                        wait_acc();
                        uint32_t r[32];
                        ptx::tmem_ld32(t_row + (uint32_t)c0, r);
                        ptx::tmem_ld_wait();
                        uint32_t *srow = reinterpret_cast<uint32_t *>(xpose) + lane * TC_XPOSE_PITCH;
#pragma unroll
                        for (int j = 0; j < 32; j++) srow[j] = r[j];
                        __syncwarp();
                        float ysum[8];                             // (sum, sum of squares) of this lane's rows for its 4 channels (y_part)
                        if (rows_ok) {
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                const int c = cq + 8 * j;
                                const float bias = e.bias ? __ldg(e.bias + col0 + c) : 0.f;
                                const float *sc = xpose + (8 * rg) * TC_XPOSE_PITCH + c;
                                const uint32_t xw[4] = {xin[j].x, xin[j].y, xin[j].z, xin[j].w};
                                uint32_t o[4];
#pragma unroll
                                for (int i = 0; i < 4; i++)
                                    o[i] = pack_bf16x2(sc[(2 * i) * TC_XPOSE_PITCH] + bias + bf16_lo(xw[i]),
                                                       sc[(2 * i + 1) * TC_XPOSE_PITCH] + bias + bf16_hi(xw[i]));
                                *reinterpret_cast<uint4 *>(yrow + (int64_t)(col0 + c) * e.ysc) = make_uint4(o[0], o[1], o[2], o[3]);
                                if (e.y_part != nullptr) {      // statistics of y AS STORED: this lane's 8 rows of channel c
                                    float s1 = 0.f, s2 = 0.f;
#pragma unroll
                                    for (int i = 0; i < 4; i++) {
                                        const float y0 = bf16_lo(o[i]), y1 = bf16_hi(o[i]);
                                        s1 += y0 + y1; s2 = fmaf(y0, y0, fmaf(y1, y1, s2));
                                    }
                                    ysum[2 * j] = s1; ysum[2 * j + 1] = s2;
                                }
                            }
                            if (e.y_part != nullptr) {
                                // the 4 lanes (rg) that share a channel column: reduce-scatter, lane rg ends with the totals of channel
                                // cq + 8 * rg -> one (sum, sum of squares) per 32-row block and channel, no atomics
                                lane_group_reduce_scatter<8, 4>(ysum, lane);
                                e.y_part[(row0 >> 5) * e.N + col0 + cq + 8 * rg] = make_float2(ysum[0], ysum[1]);
                            }
                        }
                        __syncwarp();
                    }
                } else {
                    // generic (ragged P / unaligned) path: one position per lane, 2-byte accesses coalesced along p
                    wait_acc();
                    const int64_t row = row0 + lane;
                    for (int c0 = half * 32; c0 < p.block_n; c0 += 64) {
#pragma unroll
                        for (int hc = 0; hc < 2; hc++) {
                            uint32_t r[16];
                            ptx::tmem_ld16(t_row + (uint32_t)(c0 + 16 * hc), r);
                            ptx::tmem_ld_wait();
                            const int col0 = n_blk * p.block_n + c0 + 16 * hc;
                            if (row < p.M && col0 < p.N) {
                                float acc[16];
#pragma unroll
                                for (int j = 0; j < 16; j++) acc[j] = __uint_as_float(r[j]);
                                epilogue_apply<EPI, std::conditional_t<(PL > 1), float, bf16>, 16>(e, row, col0, acc);
                            }
                        }
                    }
                }
            } else if constexpr (EPI == NMM_EPI_GEGLU) {
                // 64 accumulator columns (32 value/gate pairs) per chunk -> 32 bf16 outputs per row -> one 32 x 32 bf16 box
                for (int c0 = half * 64; c0 < p.block_n; c0 += 128) {
                    const int col0 = n_blk * p.block_n + c0;
                    wait_acc();
                    uint32_t o[16];
                    uint32_t olo[PL > 1 ? 16 : 1];                         // PL 2: bf16 residuals of the outputs (the lo plane); PL 3: the mid plane
                    uint32_t olo2[PL == 3 ? 16 : 1];                       // PL 3: the lo plane
                    // both 32-column halves are requested before the single tcgen05.wait::ld: one exposed TMEM latency per chunk
                    uint32_t r[2][32];
                    ptx::tmem_ld32(t_row + (uint32_t)c0, r[0]);
                    ptx::tmem_ld32(t_row + (uint32_t)(c0 + 32), r[1]);
                    auto half_chunk = [&](auto HAS_BIAS, int hc) {
                        float4 b4[8];
                        if constexpr (decltype(HAS_BIAS)::value) {
#pragma unroll
                            for (int j = 0; j < 8; j++) b4[j] = __ldg(reinterpret_cast<const float4 *>(e.bias + col0 + 32 * hc) + j);
                        }
                        if (hc == 0) ptx::tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            // accumulator columns 4j .. 4j+3 = value 2q, value 2q+1, gate 2q, gate 2q+1 (packing order, api.cu)
                            float v0, g0, v1, g1;
                            if (ln_in) {      // out = rstd * (acc - mean * g[n]) + c[n]
                                const float4 gg = __ldg(reinterpret_cast<const float4 *>(e.ln_g + col0 + 32 * hc) + j);
                                const float4 cc = __ldg(reinterpret_cast<const float4 *>(e.ln_c + col0 + 32 * hc) + j);
                                v0 = fmaf(ln_rstd, __uint_as_float(r[hc][4 * j]) - ln_mu * gg.x, cc.x);
                                v1 = fmaf(ln_rstd, __uint_as_float(r[hc][4 * j + 1]) - ln_mu * gg.y, cc.y);
                                g0 = fmaf(ln_rstd, __uint_as_float(r[hc][4 * j + 2]) - ln_mu * gg.z, cc.z);
                                g1 = fmaf(ln_rstd, __uint_as_float(r[hc][4 * j + 3]) - ln_mu * gg.w, cc.w);
                            } else if constexpr (decltype(HAS_BIAS)::value) {
                                // (v0, v1) and (g0, g1) are register-adjacent pairs of the TMEM load and of the bias vector: packed adds
                                f32x2_unpack(f32x2_add(f32x2_pack(__uint_as_float(r[hc][4 * j]), __uint_as_float(r[hc][4 * j + 1])), f32x2_pack(b4[j].x, b4[j].y)), v0, v1);
                                f32x2_unpack(f32x2_add(f32x2_pack(__uint_as_float(r[hc][4 * j + 2]), __uint_as_float(r[hc][4 * j + 3])), f32x2_pack(b4[j].z, b4[j].w)), g0, g1);
                            } else {
                                v0 = __uint_as_float(r[hc][4 * j]); v1 = __uint_as_float(r[hc][4 * j + 1]);
                                g0 = __uint_as_float(r[hc][4 * j + 2]); g1 = __uint_as_float(r[hc][4 * j + 3]);
                            }
                            float y0, y1;
                            geglu_pair(v0, g0, v1, g1, y0, y1);
                            if constexpr (PL == 3) split3_bf16x2(y0, y1, o[8 * hc + j], olo[8 * hc + j], olo2[8 * hc + j]);
                            else if constexpr (PL == 2) split_bf16x2(y0, y1, o[8 * hc + j], olo[8 * hc + j]);
                            else o[8 * hc + j] = pack_bf16x2(y0, y1);
                        }
                    };
                    if (e.bias != nullptr && !ln_in) { half_chunk(std::true_type{}, 0); half_chunk(std::true_type{}, 1); }
                    else { half_chunk(std::false_type{}, 0); half_chunk(std::false_type{}, 1); }
                    if (lane == 0) ptx::bulk_wait_read0();                // the box of the previous chunk has been read
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 4; j++) sts128(box_bf16_addr(box0, lane, j), o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                    if constexpr (PL > 1) {
#pragma unroll
                        for (int j = 0; j < 4; j++) sts128(box_bf16_addr(box1, lane, j), olo[4 * j], olo[4 * j + 1], olo[4 * j + 2], olo[4 * j + 3]);
                    }
                    if constexpr (PL == 3) {      // the third box of the 12 KB per-warp buffer (host: epi_buf)
#pragma unroll
                        for (int j = 0; j < 4; j++) sts128(box_bf16_addr(box2, lane, j), olo2[4 * j], olo2[4 * j + 1], olo2[4 * j + 2], olo2[4 * j + 3]);
                    }
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_store_2d(&tm_o, box0, col0 / 2, (int32_t)row0);
                        if constexpr (PL > 1) ptx::tma_store_2d(&tm_o, box1, p.N / 2 + col0 / 2, (int32_t)row0);      // lo (PL 3: mid) plane: columns [N/2, N) of `out`
                        if constexpr (PL == 3) ptx::tma_store_2d(&tm_o, box2, p.N + col0 / 2, (int32_t)row0);         // PL 3: lo plane, columns [N, 3N/2)
                        ptx::bulk_commit();
                    }
                    if (warp == 4 && lane == 0 && c0 / 128 < 4) TRACE(tile_no, 8 + c0 / 128);
                }
            } else {
                // STORE / RESIDUAL: 32-column chunks.  RESIDUAL: the fp32 residual chunk is TMA-loaded into box (k & 1) one chunk
                // ahead, summed in place and TMA-stored from the same box (or written as bf16 into the box when only `out` is wanted).
                // (Measured alternative, round 2: residual rows loaded straight into registers -- lane = row, 8 x 16-byte loads per chunk,
                //  two-box store ring, no load boxes -- is 35 % SLOWER (to_out 26.8 -> 36.2 us at C = 640): 32 rows x 16 B per instruction
                //  touches 32 cache lines, and with 200+ KB of shared memory configured there is no L1 left to merge the sector halves.)
                const int first = half * 32;
                int k = 0;
                if constexpr (EPI == NMM_EPI_RESIDUAL) {
                    if (lane == 0 && first < p.block_n) {
                        ptx::bulk_wait_read0();
                        ptx::mbar_expect_tx(load_bar(ew, 0), 4096u);
                        ptx::tma_load_2d(&tm_h, load_bar(ew, 0), box0, n_blk * p.block_n + first, (int32_t)row0);
                    }
                }
                for (int c0 = first; c0 < p.block_n; c0 += 64, k++) {
                    const int col0 = n_blk * p.block_n + c0;
                    const uint32_t box = (EPI == NMM_EPI_RESIDUAL && (k & 1)) ? box1 : box0;
                    if constexpr (EPI == NMM_EPI_RESIDUAL) {
                        if (lane == 0 && c0 + 64 < p.block_n) {           // next chunk's residual into the other box
                            ptx::bulk_wait_read0();                       // ... once the store that used it has been read
                            const int nb = (k + 1) & 1;
                            ptx::mbar_expect_tx(load_bar(ew, nb), 4096u);
                            ptx::tma_load_2d(&tm_h, load_bar(ew, nb), nb ? box1 : box0, col0 + 64, (int32_t)row0);
                        }
                    }
                    wait_acc();
                    uint32_t r[32];
                    ptx::tmem_ld32(t_row + (uint32_t)c0, r);
                    ptx::tmem_ld_wait();
                    float v[32];
                    if (ln_in) {              // out = rstd * (acc - mean * g[n]) + c[n] (+ pe[frame] . W^T)
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const float4 gg = __ldg(reinterpret_cast<const float4 *>(e.ln_g + col0) + j);
                            float4 cc = __ldg(reinterpret_cast<const float4 *>(e.ln_c + col0) + j);
                            if (pew_row != nullptr) {
                                const float4 pw = __ldg(reinterpret_cast<const float4 *>(pew_row + col0) + j);
                                cc.x += pw.x; cc.y += pw.y; cc.z += pw.z; cc.w += pw.w;
                            }
                            v[4 * j] = fmaf(ln_rstd, __uint_as_float(r[4 * j]) - ln_mu * gg.x, cc.x);
                            v[4 * j + 1] = fmaf(ln_rstd, __uint_as_float(r[4 * j + 1]) - ln_mu * gg.y, cc.y);
                            v[4 * j + 2] = fmaf(ln_rstd, __uint_as_float(r[4 * j + 2]) - ln_mu * gg.z, cc.z);
                            v[4 * j + 3] = fmaf(ln_rstd, __uint_as_float(r[4 * j + 3]) - ln_mu * gg.w, cc.w);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (e.bias != nullptr) b4 = __ldg(reinterpret_cast<const float4 *>(e.bias + col0) + j);
                            v[4 * j] = __uint_as_float(r[4 * j]) + b4.x; v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b4.y;
                            v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b4.z; v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b4.w;
                        }
                    }
                    if constexpr (EPI == NMM_EPI_RESIDUAL) {
                        if (k & 1) { ptx::mbar_wait(load_bar(ew, 1), lph1); lph1 ^= 1u; }
                        else { ptx::mbar_wait(load_bar(ew, 0), lph0); lph0 ^= 1u; }
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const float4 h4 = lds128(box_f32_addr(box, lane, j));
                            v[4 * j] += h4.x; v[4 * j + 1] += h4.y; v[4 * j + 2] += h4.z; v[4 * j + 3] += h4.w;
                        }
                        if (e.out != nullptr && (PL == 3 || !e.no_h_store) && lane == 0) ptx::bulk_wait_read0();   // third box (bf16 copy; PL 3: lo plane) free again
                        __syncwarp();                                     // every lane has read its row before the box is overwritten
                    } else {
                        if (lane == 0) ptx::bulk_wait_read0();            // the previous chunk's boxes have been read
                        __syncwarp();
                    }
                    const bool want_o = e.out != nullptr;
                    const bool want_h = e.h != nullptr && !e.no_h_store;
                    if (LNF && e.ln_part_out != nullptr) {                // producer side of the LayerNorm folding
#pragma unroll
                        for (int j = 0; j < 32; j++) { st1 += v[j]; st2 = fmaf(v[j], v[j], st2); }
                    }
                    // fp32 result -> `box` (128-byte rows); bf16 result -> box1 for STORE; for RESIDUAL the consumed residual box
                    // itself when h is not stored, else the third box (host sizes the per-warp buffer accordingly)
                    const uint32_t obox = (EPI == NMM_EPI_RESIDUAL) ? (want_h ? box2 : box) : box1;
                    if (want_h) {
#pragma unroll
                        for (int j = 0; j < 8; j++)
                            sts128(box_f32_addr(box, lane, j), __float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                                   __float_as_uint(v[4 * j + 3]));
                    }
                    if (want_o) {
                        if constexpr (PL == 3) {                          // hi plane -> obox, mid plane -> obox + 2 KB, lo plane -> box2 (host: epi_buf 12 KB)
                            uint32_t hi[16], mid[16], lo[16];
#pragma unroll
                            for (int j = 0; j < 16; j++) split3_bf16x2(v[2 * j], v[2 * j + 1], hi[j], mid[j], lo[j]);
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                sts128(box_bf16_addr(obox, lane, j), hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
                                sts128(box_bf16_addr(obox + 2048u, lane, j), mid[4 * j], mid[4 * j + 1], mid[4 * j + 2], mid[4 * j + 3]);
                                sts128(box_bf16_addr(box2, lane, j), lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
                            }
                        } else if constexpr (PL == 2) {                   // hi plane -> obox, lo plane -> obox + 2 KB (both halves of a 4 KB box)
                            uint32_t hi[16], lo[16];
#pragma unroll
                            for (int j = 0; j < 16; j++) split_bf16x2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                sts128(box_bf16_addr(obox, lane, j), hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
                                sts128(box_bf16_addr(obox + 2048u, lane, j), lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; j++)
                                sts128(box_bf16_addr(obox, lane, j), pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                                       pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
                        }
                    }
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (want_h) ptx::tma_store_2d(&tm_h, box, col0, (int32_t)row0);
                        if (want_o) ptx::tma_store_2d(&tm_o, obox, col0, (int32_t)row0);
                        if constexpr (PL > 1) { if (want_o) ptx::tma_store_2d(&tm_o, obox + 2048u, p.N + col0, (int32_t)row0); }   // lo (PL 3: mid) plane: columns [N, 2N)
                        if constexpr (PL == 3) { if (want_o) ptx::tma_store_2d(&tm_o, box2, 2 * p.N + col0, (int32_t)row0); }      // PL 3: lo plane, columns [2N, 3N)
                        ptx::bulk_commit();
                    }
                    if (warp == 4 && lane == 0 && k < 4) TRACE(tile_no, 8 + k);
                }
            }
            wait_acc();                                                   // a warp without a chunk in this tile still follows the phases
            if (LNF && e.ln_part_out != nullptr && row0 + lane < p.M)     // slot = (N tile, which warp of the quadrant); zeros if no chunk
                reinterpret_cast<float2 *>(e.ln_part_out)[(row0 + lane) * (2 * p.n_tiles) + n_blk * 2 + half] = make_float2(st1, st2);
            if (warp == 4 && lane == 0) TRACE(tile_no, 12);
            if (warp == 8 && lane == 0) TRACE(tile_no, 14);
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 1) ptx::mbar_arrive(tempty_bar(as));
                else ptx::mbar_arrive_cluster(tempty_bar(as) & ptx::PEER_MASK);      // the even CTA's barrier
            }
            if (p.wide) aphase ^= 1u;
            else if (++as == 2) { as = 0; aphase ^= 1u; }
        }
        if (lane == 0) ptx::bulk_wait_all();                              // all TMA stores of this warp have completed
    }
    __syncwarp();                                    // lanes 1-31 of the single-thread roles rejoin lane 0 before the aligned barrier
    ptx::tc_fence_before();
    if (CG > 1) ptx::cluster_sync();                 // the peer may still read this CTA's shared memory / arrive on its barriers
    else __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<CG>(tmem_base, (uint32_t)p.tmem_cols);
    }
}

// ---- host side ----------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// [rows, cols] row-major tensor with leading dimension ld (elements); box = box_rows x box_cols.
static int make_tmap(CUtensorMap *tm, const void *ptr, CUtensorMapDataType dt, int esize, int64_t rows, int64_t cols, int64_t ld,
                     int box_rows, int box_cols, CUtensorMapSwizzle swz) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(NMM_ERR_DEVICE, "cuTensorMapEncodeTiled not available (no CUDA driver?)");
    if (!aligned(ptr, 16) || (ld * esize) % 16 != 0) return fail(NMM_ERR_BAD_ARG, "TMA operand must be 16-byte aligned with a 16-byte multiple row pitch");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * esize};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(tm, dt, 2, const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NMM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return NMM_OK;
}

// x [B, C, F, P] (element strides sb, sc, sf; unit stride along P) as a 4-D tensor (p, c, f, b); box = 64 positions x 64 channels.
static int make_tmap_x(CUtensorMap *tm, const void *x, int B, int C, int F, int P, int64_t sb, int64_t sc, int64_t sf) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(NMM_ERR_DEVICE, "cuTensorMapEncodeTiled not available (no CUDA driver?)");
    cuuint64_t dims[4] = {(cuuint64_t)P, (cuuint64_t)C, (cuuint64_t)F, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)sc * 2, (cuuint64_t)sf * 2, (cuuint64_t)sb * 2};
    cuuint32_t box[4] = {64, 64, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NMM_ERR_CUDA, "cuTensorMapEncodeTiled (x, 4-D) failed with CUresult %d", (int)r);
    return NMM_OK;
}

// tokens [B*F*P, C] viewed as (c, b*F + f, p) -- note the dimension ORDER: frames before positions, so that a box of
// (64 channels, F frames, 128/F positions) lands in shared memory as rows pl * F + f, the attention tile order.
static int make_tmap_tokens_pf(CUtensorMap *tm, const void *tok, int B, int C, int F, int P, int ppt) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(NMM_ERR_DEVICE, "cuTensorMapEncodeTiled not available (no CUDA driver?)");
    cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)B * F, (cuuint64_t)P};
    cuuint64_t strides[2] = {(cuuint64_t)P * C * 2, (cuuint64_t)C * 2};
    cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)F, (cuuint32_t)ppt};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(tok), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NMM_ERR_CUDA, "cuTensorMapEncodeTiled (tokens, 3-D) failed with CUresult %d", (int)r);
    return NMM_OK;
}

// Can the temporal attention run inside the QKV projection's epilogue?  See LinearArgs (NMM_EPI_QKV_ATTN).
bool linear_tc_attn_fusable(int C, int heads, int F, int P) {
    if (heads <= 0 || C % heads != 0 || C % NMM_ATTN_TILE_CH != 0) return false;
    const int dh = C / heads;
    return (dh == 40 || dh == 80) && (F == 8 || F == 16) && P % (TC_BM / F) == 0 && opt(NMM_OPT_ATTN_FUSE) != 0;
}

// Can proj_in take its A operand straight from x (GroupNorm applied in shared memory)?  See LinearArgs::gn_x.
bool linear_tc_gn_fusable(int64_t M, int P, const void *x, int64_t sb, int64_t sc, int64_t sf) {
    return P % 64 == 0 && M % TC_BM == 0 && aligned(x, 16) && sb % 8 == 0 && sc % 8 == 0 && sf % 8 == 0 && opt(NMM_OPT_GN_FUSE) != 0;
}

#ifdef NMM_TRACE
static unsigned long long *g_trace_dev = nullptr;
extern "C" __attribute__((visibility("default"))) int nmm_debug_trace_dump(const char *path) {
    if (!g_trace_dev) return -1;
    static unsigned long long host[TRACE_TILES * TRACE_SLOTS];
    cudaDeviceSynchronize();
    cudaMemcpy(host, g_trace_dev, sizeof(host), cudaMemcpyDeviceToHost);
    FILE *f = fopen(path, "w");
    if (!f) return -2;
    for (int t = 0; t < TRACE_TILES; t++) {
        for (int s = 0; s < TRACE_SLOTS; s++) fprintf(f, "%llu ", host[t * TRACE_SLOTS + s]);
        fprintf(f, "\n");
    }
    fclose(f);
    cudaMemset(g_trace_dev, 0, sizeof(host));
    return 0;
}
#endif

static int num_sms() {                 // SM count of the CURRENT device (cached per ordinal)
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    int n = cache[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cache[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

// Tile selection.  Candidates: N tile = a multiple of `gran` (32; 64 for GEGLU, whose chunks are 64 accumulator columns) in
// [gran, 256] that divides N, x CTAs per tile CG in {1, 2}.  Cost model (cycles, from the measurements in the file header):
//   per k-block   max( MMA: 2*bn ,  operand fill: (16 KB + bn*128/CG bytes) / 64 B/clk of per-SM TMA ingest )
//   per tile      num_kb * that + a fixed per-tile overhead (barrier round trips, epilogue tail)
//   whole GEMM    ceil(cluster_tiles / resident clusters) * per tile            (wave quantisation)
// The per-SM ingest of ~64 B/clk is why only (CG = 2, bn = 256) can keep the tensor pipe fully fed, and why small tiles lose.
struct TilePlan { int block_n, cluster, wide; };
static TilePlan choose_tiles(int64_t m_tiles, int N, int K, int sms, int gran, int force_cluster, int force_bn, bool allow_wide = false,
                             int max_bn = 256) {
    TilePlan best = {0, 1, 0};
    double best_cost = 1e300;
    const int num_kb = (K + TC_BK - 1) / TC_BK;
    for (int cg = 1; cg <= 2; cg++) {
        if (force_cluster && cg != force_cluster) continue;
        if (cg == 2 && (m_tiles < 2 || sms % 2 != 0)) continue;
        const int64_t m_groups = ceil_div(m_tiles, cg);
        for (int bn = max_bn / gran * gran; bn >= gran; bn -= gran) {
            if (N % bn) continue;
            if (force_bn && bn != force_bn) continue;
            const double mma = 2.0 * bn, fill = (16384.0 + bn * 128.0 / cg) / 64.0;
            // + per-tile overhead; a CTA pair also pays for keeping two CTAs in lock-step (measured: pairs lose for K = 320)
            const double per_tile = num_kb * (mma > fill ? mma : fill) + 1500.0 + 4.0 * bn + (cg == 2 ? (num_kb <= 10 ? 2500.0 : 1500.0) : 0.0);
            const int64_t cluster_tiles = m_groups * (N / bn);
            const int64_t resident = sms / cg;
            const double cost = (double)ceil_div(cluster_tiles, resident) * per_tile;
            if (cost < best_cost) { best_cost = cost; best.block_n = bn; best.cluster = cg; best.wide = 0; }
        }
    }
    // Wide pair tile: 256 x 320 per CTA pair as two N = 160 MMAs per k-step into one 320-column accumulator.  Per CTA and k-block
    // 16 KB of A + 20 KB of W feed 128 x 320 outputs (1.45x the arithmetic intensity of 256 x 160), but with a single accumulator the
    // epilogue (~16 cycles per column) is not hidden behind the next tile's MMAs: it pays for long K and few waves (ff_out).
    // (K >= 1280 only: measured at K = 640 -- to_out of the C = 640 level -- the exposed epilogue loses: 39.1 us against 34.4 us for 128 x 160 tiles)
    if (allow_wide && num_kb >= 20 && N % 320 == 0 && sms % 2 == 0 && m_tiles >= 2 && force_cluster != 1 && (force_bn == 0 || force_bn == 320)) {
        const double mma = 2.0 * 320, fill = (16384.0 + 320 * 128.0 / 2) / 64.0;
        const double per_tile = num_kb * (mma > fill ? mma : fill) + 3000.0 + 20.0 * 320;
        const double cost = (double)ceil_div(ceil_div(m_tiles, 2) * (N / 320), (int64_t)(sms / 2)) * per_tile;
        if (cost < best_cost || force_bn == 320) { best_cost = cost; best.block_n = 320; best.cluster = 2; best.wide = 1; }
    }
    return best;
}

void plan_linear_tc(int64_t M, int N, int K, int epilogue, int *block_n, int *cluster) {
    const int force_cluster = (int)opt(NMM_OPT_GEMM_CLUSTER), force_bn = (int)opt(NMM_OPT_GEMM_BLOCK_N);
    const int gran = epilogue == NMM_EPI_GEGLU ? 64 : 32;
    const TilePlan plan = choose_tiles(ceil_div(M, TC_BM), N, K, num_sms(), gran, (force_cluster == 1 || force_cluster == 2) ? force_cluster : 0,
                                       (force_bn >= gran && force_bn <= 256 && force_bn % gran == 0 && N % force_bn == 0) ? force_bn : 0);
    *block_n = plan.block_n;
    *cluster = plan.cluster;
}

template <int EPI, int CG, bool LNF, bool GNA = false, int PL = 1>
static int launch_tc_t(const CUtensorMap &ta, const CUtensorMap &tw, const CUtensorMap &th, const CUtensorMap &to, const TcParams &p,
                       const EpiParams &e, size_t smem, int grid, cudaStream_t st, double flops, double bytes, const GnParams &gn = GnParams(),
                       const AttnParams &at = AttnParams()) {
    auto kern = linear_tc_kernel<EPI, CG, LNF, GNA, PL>;
    static DeviceOnce once;           // per template instantiation and device
    NMM_CUDA_OK(once.max_smem(kern, TC_SMEM_MAX));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(EPI == NMM_EPI_QKV_ATTN ? TC_THREADS + 32 * TC_ATTN_HELPERS : GNA ? TC_THREADS + 32 * TC_GN_WARPS : TC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = (unsigned)CG;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = CG > 1 ? 2 : 1;
    {
        ProfScope prof(K_LINEAR_TC, st, flops, bytes);
        cudaError_t le = cudaLaunchKernelEx(&cfg, kern, ta, tw, th, to, p, e, gn, at);
        if (le != cudaSuccess) return fail(NMM_ERR_CUDA, "cudaLaunchKernelEx(linear_tc_kernel) failed: %s", cudaGetErrorString(le));
    }
    NMM_LAUNCHED("linear_tc_kernel");
    return NMM_OK;
}

int launch_linear_tc(const LinearArgs &a, cudaStream_t st) {
    if (a.N % 32 != 0) return fail(NMM_ERR_UNSUPPORTED, "tcgen05 GEMM needs N %% 32 == 0 (N=%d)", a.N);
    if (a.epilogue == NMM_EPI_GEGLU && a.N % 64 != 0) return fail(NMM_ERR_UNSUPPORTED, "GEGLU epilogue needs N %% 64 == 0 (N=%d)", a.N);
    if (a.K % 8 != 0) return fail(NMM_ERR_UNSUPPORTED, "tcgen05 GEMM needs K %% 8 == 0 (K=%d)", a.K);
    const int planes = a.planes > 1 ? a.planes : 1;
    if (planes > 3) return fail(NMM_ERR_BAD_ARG, "tcgen05 GEMM: %d operand planes (1, 2 or 3)", planes);
    const bool x3 = planes > 1;
    if (x3 && (a.K % TC_BK != 0 || a.gn_x != nullptr || a.epilogue == NMM_EPI_QKV_ATTN || a.ln_part_in != nullptr || a.ln_part_out != nullptr ||
               (a.epilogue == NMM_EPI_STORE && a.out != nullptr) || (a.epilogue == NMM_EPI_RESIDUAL && a.out != nullptr && !a.no_h_store)))
        return fail(NMM_ERR_UNSUPPORTED, "3 / 6 x bf16 (fp32-grade / fp32-exact) tensor-core GEMM: needs K %% 64 == 0, no fused GroupNorm / attention / LayerNorm folding, and a STORE epilogue writing fp32 only");
    if (a.M <= 0) return NMM_OK;
    TcParams p;
    p.M = a.M; p.N = a.N; p.K = a.K;
    p.m_tiles = ceil_div(a.M, TC_BM);
    const int sms = num_sms();
    // NMM_OPT_GEMM_CLUSTER / NMM_OPT_GEMM_BLOCK_N force a tiling (development).  The result-invalidating timing experiments
    // (NMM_GEMM_DEBUG: epilogue off / no TMA loads / ...) exist only in the -DNMM_TRACE development build.
#ifdef NMM_TRACE
    static const int debug_flags = getenv("NMM_GEMM_DEBUG") ? atoi(getenv("NMM_GEMM_DEBUG")) : 0;
#else
    constexpr int debug_flags = 0;
#endif
    // (the no-TMA timing experiment is only wired for single-CTA tiles)
    const int force_cluster = (debug_flags & 2) ? 1 : (int)opt(NMM_OPT_GEMM_CLUSTER);
    const int force_bn = (int)opt(NMM_OPT_GEMM_BLOCK_N);
    p.debug = debug_flags;
    p.trace = nullptr;
    p.chunk_kb = planes == 3 ? TC_X6_CHUNK_KB : 0;
#ifdef NMM_TRACE
    if (!g_trace_dev) { cudaMalloc(&g_trace_dev, TRACE_TILES * TRACE_SLOTS * 8); cudaMemset(g_trace_dev, 0, TRACE_TILES * TRACE_SLOTS * 8); }
    p.trace = g_trace_dev;
#endif
    const bool attn = a.epilogue == NMM_EPI_QKV_ATTN;
    if (attn && (a.out == nullptr || a.A == nullptr || a.N != 3 * a.K || a.attn_B <= 0 || !linear_tc_attn_fusable(a.K, a.attn_heads, a.F, a.P) ||
                 (int64_t)a.attn_B * a.F * a.P != a.M || a.ln_part_in != nullptr || a.ln_part_out != nullptr || a.gn_x != nullptr))
        return fail(NMM_ERR_UNSUPPORTED, "fused QKV + attention: needs d_h in {40, 80}, F in {8, 16}, P %% (128 / F) == 0");
    const bool gna = a.gn_x != nullptr;
    if (gna && (a.epilogue != NMM_EPI_STORE || a.ln_part_in != nullptr || a.ln_part_out != nullptr || a.gn_B <= 0 ||
                !linear_tc_gn_fusable(a.M, a.P, a.gn_x, a.xsb, a.xsc, a.xsf) || (int64_t)a.gn_B * a.F * a.P != a.M))
        return fail(NMM_ERR_UNSUPPORTED, "GroupNorm-fused A operand: needs the STORE epilogue, P %% 64 == 0, M %% 128 == 0 and 16-byte aligned x");
    const int gran = a.epilogue == NMM_EPI_GEGLU ? 64 : 32;
    const bool allow_wide = a.epilogue == NMM_EPI_RESIDUAL && planes != 3 && !gna && a.ln_part_in == nullptr && a.ln_part_out == nullptr && !(debug_flags & 2) && opt(NMM_OPT_WIDE_TILE) != 0;
    const TilePlan plan = attn ? TilePlan{3 * NMM_ATTN_TILE_CH, 1, 0} :
                          choose_tiles(p.m_tiles, a.N, (planes == 3 ? 6 : planes == 2 ? 3 : 1) * a.K, sms, gran, gna ? 1 : (force_cluster == 1 || force_cluster == 2) ? force_cluster : 0,
                                       (force_bn >= gran && force_bn <= (planes == 3 ? TC_X6_MAX_BN : 320) && force_bn % gran == 0 && a.N % force_bn == 0) ? force_bn : 0,
                                       allow_wide, planes == 3 ? TC_X6_MAX_BN : 256);
    if (plan.block_n == 0) return fail(NMM_ERR_UNSUPPORTED, "tcgen05 GEMM: no N tile for N=%d", a.N);
    p.block_n = plan.block_n;
    p.cluster = plan.cluster;
    p.wide = plan.wide;
    const int64_t m_groups = ceil_div(p.m_tiles, p.cluster);
    p.n_tiles = a.N / p.block_n;
    p.cluster_tiles = m_groups * p.n_tiles;
    const size_t stage_bytes = (size_t)TC_A_BYTES + (size_t)(p.block_n / p.cluster) * TC_BK * 2;     // per CTA
    // a third 4 KB box: RESIDUAL writing h and a bf16 copy; PL 3 writing a third plane (GEGLU, RESIDUAL with `out`)
    p.epi_buf = ((a.epilogue == NMM_EPI_RESIDUAL && a.out != nullptr && !a.no_h_store) ||
                 (planes == 3 && a.out != nullptr && (a.epilogue == NMM_EPI_GEGLU || a.epilogue == NMM_EPI_RESIDUAL))) ? 12288 : TC_EPI_BUF;
    const size_t gn_coef = a.gn_x != nullptr ? (size_t)ceil_div(a.K, TC_BK) * TC_BK * 8 : 0;      // GNA: gamma | beta in shared memory
    const size_t fixed = 1024 /*alignment slack*/ + TC_BAR_BYTES + (size_t)TC_EPI_WARPS * p.epi_buf + gn_coef;
    int stages = (int)((TC_SMEM_MAX - fixed) / stage_bytes);
    if (stages > 8) stages = 8;
    if (stages < 2) return fail(NMM_ERR_UNSUPPORTED, "tcgen05 GEMM: tile does not fit shared memory");
    p.stages = stages;
    int cols = 32;
    while (cols < (p.wide ? 1 : 2) * p.block_n) cols <<= 1;       // wide tiles keep one accumulator
    p.tmem_cols = cols;
    const size_t smem = fixed + (size_t)stages * stage_bytes;
    CUtensorMap ta, tw, th, to;
    const int64_t kcols = planes * (int64_t)a.K;                 // PL > 1: [hi | lo] / [hi | mid | lo] planes side by side
    int rc = attn ? make_tmap_tokens_pf(&ta, a.A, a.attn_B, a.K, a.F, a.P, TC_BM / a.F)
             : gna ? make_tmap_x(&ta, a.gn_x, a.gn_B, a.K, a.F, a.P, a.xsb, a.xsc, a.xsf)
                 : make_tmap(&ta, a.A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a.M, kcols, kcols, TC_BM, TC_BK, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != NMM_OK) return rc;
    // each CTA of a pair fetches its slice of the W tile
    rc = make_tmap(&tw, a.W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a.N, kcols, kcols, p.block_n / p.cluster / (p.wide ? 2 : 1), TC_BK, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != NMM_OK) return rc;
    memset(&th, 0, sizeof(th));
    memset(&to, 0, sizeof(to));
    if (a.h != nullptr && a.epilogue != NMM_EPI_OUTPUT && a.epilogue != NMM_EPI_GEGLU) {
        rc = make_tmap(&th, a.h, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.M, a.N, a.N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc != NMM_OK) return rc;
    }
    if (a.out != nullptr && a.epilogue != NMM_EPI_OUTPUT && !attn) {
        const int64_t ncols = (a.epilogue == NMM_EPI_GEGLU ? a.N / 2 : a.N) * planes;
        rc = make_tmap(&to, a.out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a.M, ncols, ncols, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
        if (rc != NMM_OK) return rc;
    }
    const int64_t ctas = p.cluster_tiles * p.cluster;
    const int max_grid = sms / p.cluster * p.cluster;
    const int grid = (int)(ctas < max_grid ? ctas : max_grid);
    EpiParams e = epi_params_of(a);
    const double fl = linear_flops(a), by = linear_bytes(a, 2);
    const bool lnf = a.ln_part_in != nullptr || a.ln_part_out != nullptr;
    if (attn) {
        AttnParams at;
        at.ctx = (bf16 *)a.out; at.C = a.K; at.F = a.F; at.P = a.P; at.dh = a.K / a.attn_heads; at.ppt = TC_BM / a.F; at.tiles_per_img = a.P / at.ppt;
        at.scale_log2e = (1.0f / sqrtf((float)at.dh)) * 1.4426950408889634f;
        // algorithmic work of the pair of kernels it replaces: the projection's FLOPs + the attention's
        return launch_tc_t<NMM_EPI_QKV_ATTN, 1, false, false>(ta, tw, th, to, p, e, smem, grid, st, fl + 4.0 * a.M * a.F * a.K, by, GnParams(), at);
    }
    if (gna) {
        GnParams gn;
        gn.partial = a.gn_partial; gn.gamma = a.gn_w; gn.beta = a.gn_b; gn.splits = a.gn_splits; gn.count = a.gn_count; gn.eps = a.gn_eps;
        gn.C = a.K; gn.F = a.F; gn.P = a.P;
        return launch_tc_t<NMM_EPI_STORE, 1, false, true>(ta, tw, th, to, p, e, smem, grid, st, fl, by, gn);
    }
#define TC_DISPATCH(EPI)                                                                                   \
    if (planes == 3)                                                                                       \
        return p.cluster == 2 ? launch_tc_t<EPI, 2, false, false, 3>(ta, tw, th, to, p, e, smem, grid, st, fl, by)       \
                              : launch_tc_t<EPI, 1, false, false, 3>(ta, tw, th, to, p, e, smem, grid, st, fl, by);      \
    if (x3)                                                                                                \
        return p.cluster == 2 ? launch_tc_t<EPI, 2, false, false, 2>(ta, tw, th, to, p, e, smem, grid, st, fl, by)       \
                              : launch_tc_t<EPI, 1, false, false, 2>(ta, tw, th, to, p, e, smem, grid, st, fl, by);      \
    if (lnf)                                                                                               \
        return p.cluster == 2 ? launch_tc_t<EPI, 2, true>(ta, tw, th, to, p, e, smem, grid, st, fl, by)    \
                              : launch_tc_t<EPI, 1, true>(ta, tw, th, to, p, e, smem, grid, st, fl, by);   \
    return p.cluster == 2 ? launch_tc_t<EPI, 2, false>(ta, tw, th, to, p, e, smem, grid, st, fl, by)       \
                          : launch_tc_t<EPI, 1, false>(ta, tw, th, to, p, e, smem, grid, st, fl, by)
    switch (a.epilogue) {
        case NMM_EPI_STORE: TC_DISPATCH(NMM_EPI_STORE);
        case NMM_EPI_RESIDUAL: TC_DISPATCH(NMM_EPI_RESIDUAL);
        case NMM_EPI_GEGLU: TC_DISPATCH(NMM_EPI_GEGLU);
        case NMM_EPI_OUTPUT: TC_DISPATCH(NMM_EPI_OUTPUT);
        default: return fail(NMM_ERR_BAD_ARG, "unknown epilogue %d", a.epilogue);
    }
#undef TC_DISPATCH
}

}  // namespace nmm

// Conv2D (1x1 and k x k, stride 1 and 2) as an implicit GEMM on Blackwell's 5th-generation tensor
// cores, hand-written for sm_100a: TMA (cp.async.bulk.tensor) stages NHWC activation tiles and packed weights from HBM
// into 128B-swizzled shared memory, one elected thread issues tcgen05.mma, accumulators live in TMEM and are read back
// with tcgen05.ld by the epilogue warps (bias + residual + activation + split-fp16 store).
//
//   D[M = 128 output pixels, N = n_blk <= 128 output channels] += A[M, K] * B[N, K]^T,   K = (tap, 64-channel block)
//
// fp32-faithful arithmetic out of fp16 tensor cores: activations and weights are stored as hi + lo fp16 pairs
// (snnb_internal.h); every K block accumulates into fp32 TMEM, template parameter TERMS:
//   3:  A_hi*B_hi + A_lo*B_hi + A_hi*B_lo   (the dropped A_lo*B_lo term is ~2^-24 relative): ~22 mantissa bits per operand. Issued
//       as TWO instructions per K=16 step: A_hi x [B_hi ; B_lo] (N = 2 n_blk, two accumulator column blocks) and A_lo x B_hi
//       (onto the first block); the epilogue adds the blocks. n_blk <= 128.
//   2:  (A_hi + A_lo) * B_hi: the weights rounded ONCE to fp16 (<= 2^-12 relative per weight, measured per-layer error vs the
//       oracle ~1e-4 of the tensor's range - inside the 1e-3 budget), two instructions, ONE accumulator block, n_blk <= 256.
//   1:  A_hi * B_hi: the half-precision storage mode (the reference's RGBA16F), no lo planes anywhere.
//
// A tile = a (tw x th x tn)-pixel box of the OUTPUT grid (tw*th*tn <= 128): for filter tap (ky,kx) the producer issues
// ONE 4-D TMA box load at input coordinate (ox0*s + kx - pad_x, oy0*s + ky - pad_y); out-of-range rows/columns are
// zero-filled by the TMA unit, which is exactly the reference's constant padding (vk_conv2d.comp:168-172), and the
// channel tail (c >= IC) is zero-filled too, so no im2col buffer and no boundary code exist anywhere.
//
// Roles (320 threads, persistent CTAs, one per SM): warp 0 = TMA producer (also draws work items from a global counter),
// warp 1 = TMEM allocator + one thread that owns the MMA issue loop, warps 2-9 = epilogue (TMEM -> registers -> swizzled smem
// -> TMA bulk store). Pipelines: smem full/empty ring and a double-buffered TMEM accumulator (tmem_full/tmem_empty), so the
// epilogue of tile i overlaps the mainloop of tile i+1. Layers with few tiles split K over several CTAs (fp32 partials, last
// arriver reduces); layers with a short K loop use two independent epilogue groups. Also in this file: the row-window kernel
// for small-channel stems and the TMA-staged depthwise kernel. DESIGN.md section 3 has the measurements behind each choice.
//
// Reference semantics: shadertemplate_vk_conv2d.comp:148-347, vk_conv2d_1x1.comp:68-211 (+ fused vk_add.comp:41-90).
#include <cuda.h>

#include <algorithm>
#include <vector>
#include <cstdlib>

#include "snnb_internal.h"

namespace snnb {

constexpr int UM_BLOCK_M     = 128;
constexpr int UM_BLOCK_K     = 64; // fp16 elements: 128 bytes = one SWIZZLE_128B row
constexpr int UM_MAX_N       = 128; // 3-term product: the accumulator holds two column blocks of n_blk
constexpr int UM_MAX_N2      = 256; // 2-term (fp16 weights) and 1-term (fp16 storage) products: one column block
constexpr int UM_STAGES      = 3;
constexpr int UM_A_BYTES     = UM_BLOCK_M * 128;
constexpr int UM_B_BYTES     = UM_MAX_N * 128;
constexpr int UM_STAGE_BYTES = 2 * UM_A_BYTES + 2 * UM_B_BYTES; // A_hi, A_lo, then [B_hi ; B_lo] (3-term) or one B plane of up to 256 rows = 64 KB
constexpr int UM_EPI_WARPS   = 8;                       // two warps per TMEM lane quarter, interleaved over 16-column chunks
constexpr int UM_THREADS     = 64 + 32 * UM_EPI_WARPS; // warp 0 TMA, warp 1 MMA, warps 2.. epilogue
constexpr int UM_ACC_COLS    = 2 * UM_MAX_N; // one accumulator buffer: [A_hi.B_hi + A_lo.B_hi | A_hi.B_lo], up to 2 x 128 fp32 columns
constexpr int UM_TMEM_COLS   = 2 * UM_ACC_COLS; // double-buffered: all 512 columns
constexpr int UM_STG_BYTES   = 2 * UM_BLOCK_M * 128; // epilogue staging: one 64-channel slab, hi + lo planes (32 KB)
constexpr int UM_SCHED_SLOTS = 8;                        // ring of work-item ids handed from the producer warp to the MMA / epilogue warps
constexpr int UM_SMEM_BYTES  = UM_STAGES * UM_STAGE_BYTES + UM_STG_BYTES + 1024 /*alignment slack*/ + 320 /*barriers + scheduler ring*/;
constexpr int UM_SMEM_BYTES_SPLIT = (UM_STAGES - 1) * UM_STAGE_BYTES + 2 * UM_STG_BYTES + 1024 + 320; // two epilogue groups, one ring stage less

// ---- halo mode (3x3, stride 1): the A operand of all nine taps comes from ONE (8+2) x (16+2)-pixel halo tile per 64-channel
// block, loaded once by TMA; tap (ky,kx) is the same shared memory read through a descriptor whose start address is shifted
// by (ky * 10 + kx) pixels and whose 8-row group stride (SBO) is the halo's row pitch, 10 pixels = 1280 B. Legal because both
// the TMA unit and the tensor core apply SWIZZLE_128B to absolute shared-memory address bits (tools/umma_desc_probe.cu), so a
// pixel row is found where TMA put it whatever the descriptor's phase. L2 -> SM traffic of A drops from 9 x 32 KB to 46 KB per
// tile and channel block (the r01 kernel moved 363-389 MB per 56x56x64 launch against 51.5 MB algorithmic: it was bound by
// the ~72 B/clk/SM the SM can ingest, not by the tensor pipe). The weights (one K block per tap) keep their own ring.
constexpr int HL_TW = 8, HL_TH = 16, HL_W = HL_TW + 2, HL_H = HL_TH + 2;
constexpr int HL_PLANE         = (HL_W * HL_H * 128 + 1023) / 1024 * 1024; // 23 552 B: one plane of the halo tile, 1024-aligned
constexpr int HL_A_STAGES      = 2;
constexpr int HL_A_STAGE_BYTES = 2 * HL_PLANE;
constexpr int HL_B_STAGES      = 6;              // == the STAGES template argument of the halo instantiations (barrier slots)
constexpr int HL_B_RING_BYTES  = 6 * UM_B_BYTES; // 96 KB of weight stages: 3 x 32 KB ([B_hi ; B_lo] of 128 rows / one plane of 256 rows) or 6 x 16 KB
constexpr int HL_SMEM_BYTES    = HL_A_STAGES * HL_A_STAGE_BYTES + HL_B_RING_BYTES + UM_STG_BYTES + 1024 + 384;

struct UmmaParams {
    __half* out_hi;
    __half* out_lo;
    const __half* res_hi;
    const __half* res_lo;
    const float* bias;
    int N, OH, OW, OC, OCp;
    int tw, th, tn, rows_used;
    int tiles_x, tiles_y, tiles_n, tiles_oc, n_blk;
    int ksize, stride, pad_x, pad_y;
    int cblocks, ICp;
    int act;
    float alpha;
    int has_res;
    // split-K (layers with too few output tiles to fill the GPU, e.g. 7x7x512): work item = (tile, K range). Every item
    // dumps its fp32 partial tile to `partials`, bumps the tile's arrival counter, and the LAST arriver sums all partials
    // in split order (deterministic) and runs the normal epilogue.
    int ksplit, kb_per_split;
    int* sched_counter; // dynamic work distribution: next work item = gridDim.x + atomicAdd(counter, 1); zero between launches
    float* partials; // [tile][split][128 rows][n_blk]
    int* counters;   // [tile], zero between launches (the last arriver resets it)
    long long* trace; // profiling aid (env SNNB_UMMA_TRACE): CTA 0 writes clock64 stamps per role, [6][256]
    int ablate; // profiling aid (env SNNB_UMMA_ABLATE, results are WRONG when set): 1 skip epilogue work, 2 skip TMA loads, 4 skip MMAs
    int has_lo; // the output tensor has a lo plane (0 in the fp16 storage mode)
    // Stream-K (sk != 0, plain mode): the first sk_dp tiles (a multiple of the grid) are whole-tile work items, CTA b taking tiles
    // b, b + grid, ...; the K-block units of the remaining tiles (sk_units = tiles x K blocks, laid end to end) are cut into sk_ctas
    // equal ranges, CTA b < sk_ctas taking range b - which covers the tail of one tile and the head of the next. A tile cut into
    // pieces is finished like a split-K tile (fp32 partials, last arriver sums them in piece order). Work ids: [0, sk_dp) tiles,
    // sk_dp + 4 c + j = the j-th piece of CTA c's range; the schedule is static (no draw from sched_counter): pieces first, then tiles.
    int sk, sk_dp, sk_ctas;
    long long sk_units;
    int b_stages, b_stage_bytes; // halo mode: depth and stage size of the weight ring (3 x 32 KB, or 6 x 16 KB when a stage fits)
    // Folded projection shortcut (plain mode only, ConvArgs::shortcut): a 1x1 stride-sc_stride convolution of another tensor onto the
    // same output grid, computed as sc_cblocks extra K blocks after the k x k taps (operand tmS_hi / tmS_lo, weight columns
    // ksize * ksize * ICp + cb * 64). sc_cblocks = 0: no shortcut.
    int sc_cblocks, sc_stride;
};

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) { // never suspends
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Progress word of every CTA's producer warp (debugging aid: printed when a wait times out)
__device__ unsigned int g_producer_progress[1024];
__device__ __forceinline__ void producer_progress(int lane, unsigned int code) {
    if (lane == 0) *reinterpret_cast<volatile unsigned int*>(&g_producer_progress[blockIdx.x & 1023]) = code;
}
// Bounded wait: a broken descriptor or protocol bug must surface as a trapped kernel, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    bool reported      = false;
    while (!mbar_try_wait(bar, parity)) {
        const long long dt = clock64() - t0;
        if (dt > 4000000000LL && !reported) {
            uint32_t dyn;
            asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
            printf("tcgen05 kernel (dynamic smem %u B): mbarrier wait timed out (block %d thread %d bar 0x%x parity %u, producer progress 0x%x)\n", dyn, blockIdx.x,
                   threadIdx.x, bar, parity, *reinterpret_cast<volatile unsigned int*>(&g_producer_progress[blockIdx.x & 1023]));
            reported = true;
        }
        if (dt > 4040000000LL) __trap(); // ~20 ms after the first report: every stuck thread gets to print
    }
}
// One lane of a CONVERGED warp. Unlike `lane == 0` the compiler knows a single thread is active in the guarded region, so
// descriptors stay in uniform registers and each tcgen05.mma / TMA issue is one predicated instruction rather than an
// ELECT + BRA.U.ANY waterfall loop (ncu r01: the issuing warp spent 77% of its time in that scalar code, not waiting).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) { asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory"); }
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst), "l"(m),
                 "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst), "l"(m), "r"(bar),
                 "r"(c0), "r"(c1)
                 : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], fp16 inputs, fp32 accumulate; issued by ONE thread for the whole CTA.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed (implicitly fences).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                   "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(m), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
// plain (non-tensor) bulk copy global -> shared, completion on an mbarrier; 16-byte aligned addresses and size
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); } // all but the newest group
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// Shared-memory matrix descriptor, K-major operand, SWIZZLE_128B (cute::UMMA::SmemDescriptor layout):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (= 1, unused for swizzled K-major) | [32,46) SBO >> 4 (= 1024 B: 8 rows x 128 B)
//   [46,48) version = 1 (Blackwell) | [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    return (uint64_t) ((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// Same with an arbitrary stride between 8-row groups (halo mode: the halo tile's row pitch, not a multiple of 1024 B)
__device__ __forceinline__ uint64_t make_smem_desc_sbo(uint32_t saddr, uint32_t sbo_bytes) {
    return (uint64_t) ((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t) (sbo_bytes >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor for kind::f16 (cute::UMMA::InstrDescriptor): c_format F32 (bit 4), a/b format at bits 7 / 10,
// both operands K-major, N >> 3 at bit 17, M >> 4 at bit 24.
// a_format / b_format (bits [7,10) / [10,13)): 0 = F16 for both operands. (kind::f16 refuses a BF16 A with an F16 B operand:
// "illegal instruction", tools/umma_desc_probe.cu - which is why the storage format is an fp16 pair, not round 1's bf16 pair.)
__device__ __forceinline__ uint32_t make_idesc(int M, int N) {
    return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t) (N >> 3) << 17) | ((uint32_t) (M >> 4) << 24);
}

// transcendental activations only (tanh / sigmoid / SiLU): rare, kept out of line so the hot epilogue stays small
__device__ __noinline__ float umma_act(float v, int act, float alpha) {
    switch (act) {
    case SNNB_ACT_RELU: return fmaxf(v, 0.0f);
    case SNNB_ACT_RELU6: return fminf(fmaxf(v, 0.0f), 6.0f);
    case SNNB_ACT_TANH: return tanhf(v);
    case SNNB_ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
    case SNNB_ACT_LEAKY_RELU: return fmaxf(v, v * alpha);
    case SNNB_ACT_SILU: return v * 1.0f / (1.0f + expf(-v));
    default: return v;
    }
}
// split-fp16 (snnb_internal.h): packed pair conversions, round to nearest, saturated to +-65504
__device__ __forceinline__ float2 um_h2f(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }
__device__ __forceinline__ uint32_t um_f2h(float a, float b) {
    uint32_t h;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(b), "f"(a));
    return h;
}
__device__ __forceinline__ void um_split2(float a, float b, uint32_t& h, uint32_t& l) {
    h               = um_f2h(a, b);
    const float2 hf = um_h2f(h);
    l               = um_f2h(a - hf.x, b - hf.y);
}

// ---------------------------------------------------------------------------------------------------------------
// Epilogue of one output tile, shared by both tensor-core kernels: TMEM -> registers -> +bias (+residual) -> activation
// -> split-fp16 -> SHARED MEMORY (128B-swizzled, bank-conflict-free) -> ONE TMA bulk store per plane and 64-channel slab.
//
// Why through smem + TMA: each thread owns one output pixel (TMEM lane), so direct global stores are 32 scattered
// 16-byte pieces per warp instruction = 32 L1 wavefronts each; at 128 rows x n_blk channels that is 8-16 k wavefronts
// per tile, MORE than the tile's MMA time - the first version of both kernels was bound by exactly that (their run time
// did not move across five different producer designs). The TMA store writes full 128-byte lines, clips rows/channels
// that fall outside the tensor by itself, and costs one instruction. The fused residual (Conv2D -> Add) comes in the same
// way: a TMA box load of the residual tile into the staging buffer, read back with swizzled LDS.
// ---------------------------------------------------------------------------------------------------------------
struct EpiArgs {
    const CUtensorMap *o_hi64, *o_lo64, *o_hiT, *o_loT; // output maps: 64-channel slab (SWIZZLE_128B) and tail slab (dense)
    const CUtensorMap *r_hi64, *r_lo64, *r_hiT, *r_loT; // residual maps, same geometry
    const float* bias;
    int n_blk, OC, act, has_res, rows_box; // 3-term: the A_hi.B_lo partial sums sit n_blk columns after the main block
    int has_lo;                            // write (and read, for the residual) the lo plane; 0 in the fp16 storage mode
    float alpha;
    uint32_t stg;       // staging smem (hi plane; lo plane at + UM_BLOCK_M * 128)
    uint32_t res_bar;   // mbarrier for the residual TMA load
    uint32_t tmem_empty;
    int bar_id;         // named barrier of this epilogue group (1, or 1 + group when two groups work on alternate tiles)
    // split-K finalisation: accumulator values come from `part_splits` fp32 partial tiles [128][n_blk] in global memory
    // (summed in split order) instead of TMEM
    const float* part_src;
    int part_splits;
    long long* trace; // profiling aid: leader warp stamps the phases of its first slabs into [4][64 + 8 * slab_seq ...]
    int trace_seq;
    bool no_store = false; // profiling aid (SNNB_UMMA_ABLATE & 8, row-window kernel): everything but the TMA store of the tile
    // Two staging buffers used on alternate tiles (row-window kernel, one slab per tile): only the store of the tile BEFORE the previous
    // one must have finished reading. The TMA store drains shared memory at ~20 B/clk per SM (1.6 k clk for a 32 KB tile,
    // profiles/r02_trace_mobilenetv2_1x1.txt); with one buffer that sat in series with the tile's arithmetic.
    bool two_stagings = false;
};

// Fused residual (Conv2D -> Add): TMA box load of the residual tile's slab into the staging buffer. The previous bulk store
// must have finished READING the buffer. Called for slab 0 BEFORE the wait for the accumulator, so the load's latency
// hides behind the tile's MMAs. `leader` is warp-uniform: the whole leader warp calls, one lane issues.
__device__ __forceinline__ void epilogue_residual_load(const EpiArgs& e, int sl, int oc0, int c1, int c2, int c3, bool leader) {
    if (!leader) return;
    const int w          = min(64, e.n_blk - sl * 64);
    const bool sw        = w == 64;
    const uint32_t pitch = sw ? 128u : (uint32_t) w * 2u;
    if (elect_one()) {
        bulk_wait_read0();
        mbar_expect_tx(e.res_bar, (e.has_lo ? 2u : 1u) * (uint32_t) e.rows_box * pitch); // the box has rows_box rows (<= 128)
        tma_load_4d(e.stg, sw ? e.r_hi64 : e.r_hiT, e.res_bar, oc0 + sl * 64, c1, c2, c3);
        if (e.has_lo) tma_load_4d(e.stg + UM_BLOCK_M * 128, sw ? e.r_lo64 : e.r_loT, e.res_bar, oc0 + sl * 64, c1, c2, c3);
    }
    __syncwarp();
}

template <int NWARPS, int TERMS>
__device__ __forceinline__ void epilogue_tile(const EpiArgs& e, uint32_t taddr, int oc0, int c1, int c2, int c3, int row, int half, bool leader, int lane,
                                              uint32_t& res_phase) {
    constexpr int MAXC  = NWARPS == 8 ? 2 : 4; // 16-column chunks of one 64-column slab owned by this warp
    const bool fast_act = e.act == SNNB_ACT_NONE || e.act == SNNB_ACT_RELU || e.act == SNNB_ACT_RELU6 || e.act == SNNB_ACT_LEAKY_RELU;
    const float slope   = (e.act == SNNB_ACT_RELU || e.act == SNNB_ACT_RELU6) ? 0.0f : (e.act == SNNB_ACT_LEAKY_RELU ? e.alpha : 1.0f);
    const float hi_clip = e.act == SNNB_ACT_RELU6 ? 6.0f : __int_as_float(0x7f800000);
    const int nslabs    = (e.n_blk + 63) >> 6;
#define EPI_STAMP(k)                                                                                      \
    do {                                                                                                  \
        if (e.trace && leader && lane == 0 && blockIdx.x == 0 && tseq < 16) e.trace[4 * 256 + 64 + 8 * tseq + (k)] = clock64(); \
    } while (0)
    for (int sl = 0; sl < nslabs; ++sl) {
        const int tseq     = e.trace_seq * nslabs + sl;
        EPI_STAMP(0);
        const int w        = min(64, e.n_blk - sl * 64); // slab width in channels (multiple of 16)
        const bool sw      = w == 64;                    // full slab: 128-byte rows, SWIZZLE_128B
        const uint32_t pitch = sw ? 128u : (uint32_t) w * 2u;
        const uint32_t srow  = e.stg + (uint32_t) row * pitch;
        const uint32_t xr    = sw ? (uint32_t) (row & 7) : 0u;
        const int slab_oc    = oc0 + sl * 64;
        if (e.has_res && sl > 0) epilogue_residual_load(e, sl, oc0, c1, c2, c3, leader); // slab 0's was issued before the accumulator wait
        // ---- phase 1: TMEM -> registers -> bias (+ residual) -> activation -> packed split-fp16, nothing written yet ----
        bool res_ready = false;
#pragma unroll
        for (int k0 = 0; k0 < MAXC; k0 += 2) { // two chunks at a time: their four TMEM loads are in flight together
            uint32_t oh[2][8], ol[2][8];
            uint32_t r[2][16], r2[2][16];
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const int ci = NWARPS == 8 ? half + 2 * (k0 + kk) : k0 + kk;
                if (ci < (w >> 4)) {
                    const int c = sl * 64 + ci * 16;
                    if (e.part_src) {
                        // all loads of the chunk are issued before the first add (L2 latency once, not once per split);
                        // summed in split order: the result does not depend on which CTA arrived last
                        float4 t[4][4];
#pragma unroll
                        for (int sp = 0; sp < 4; ++sp) {
                            // partial tile layout [chunk][j4][row][4 floats]: a warp's 32 rows are 512 contiguous bytes per access
                            const float4* src = reinterpret_cast<const float4*>(e.part_src + (size_t) sp * UM_BLOCK_M * e.n_blk) + (size_t) (c >> 4) * 4 * UM_BLOCK_M + row;
#pragma unroll
                            for (int j4 = 0; j4 < 4; ++j4)
                                t[sp][j4] = sp < e.part_splits ? __ldcg(src + j4 * UM_BLOCK_M) : make_float4(0.f, 0.f, 0.f, 0.f); // L2: written by other SMs
                        }
                        float a16[16];
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4) {
                            a16[4 * j4] = t[0][j4].x, a16[4 * j4 + 1] = t[0][j4].y, a16[4 * j4 + 2] = t[0][j4].z, a16[4 * j4 + 3] = t[0][j4].w;
#pragma unroll
                            for (int sp = 1; sp < 4; ++sp)
                                if (sp < e.part_splits) a16[4 * j4] += t[sp][j4].x, a16[4 * j4 + 1] += t[sp][j4].y, a16[4 * j4 + 2] += t[sp][j4].z, a16[4 * j4 + 3] += t[sp][j4].w;
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) r[kk][j] = __float_as_uint(a16[j]), r2[kk][j] = 0u;
                    } else {
                        tmem_ld16(taddr + (uint32_t) c, r[kk]);
                        if (TERMS == 3) {
                            tmem_ld16(taddr + (uint32_t) (e.n_blk + c), r2[kk]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) r2[kk][j] = 0u; // one column block: folded away by the compiler
                        }
                    }
                }
            }
            if (!e.part_src) tmem_ld_wait();
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const int k = k0 + kk, ci = NWARPS == 8 ? half + 2 * k : k;
                if (ci < (w >> 4)) {
                    const int c = sl * 64 + ci * 16;
                    float v[16];
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) { // the bias slice of a tile stays L1-resident across the CTA's tiles
                        const float4 b = __ldg(reinterpret_cast<const float4*>(e.bias + oc0 + c) + j4);
                        v[4 * j4 + 0] = (__uint_as_float(r[kk][4 * j4 + 0]) + __uint_as_float(r2[kk][4 * j4 + 0])) + b.x;
                        v[4 * j4 + 1] = (__uint_as_float(r[kk][4 * j4 + 1]) + __uint_as_float(r2[kk][4 * j4 + 1])) + b.y;
                        v[4 * j4 + 2] = (__uint_as_float(r[kk][4 * j4 + 2]) + __uint_as_float(r2[kk][4 * j4 + 2])) + b.z;
                        v[4 * j4 + 3] = (__uint_as_float(r[kk][4 * j4 + 3]) + __uint_as_float(r2[kk][4 * j4 + 3])) + b.w;
                    }
                    if (e.has_res) {
                        if (!res_ready) {
                            mbar_wait(e.res_bar, res_phase);
                            res_ready = true;
                        }
#pragma unroll
                        for (int g = 0; g < 2; ++g) { // this thread later overwrites exactly the 16-byte pieces it reads here
                            const uint32_t a = srow + ((((uint32_t) (ci * 2 + g)) ^ xr) << 4);
                            uint32_t hh[4], ll[4];
                            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(hh[0]), "=r"(hh[1]), "=r"(hh[2]), "=r"(hh[3]) : "r"(a));
                            if (e.has_lo) {
                                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(ll[0]), "=r"(ll[1]), "=r"(ll[2]), "=r"(ll[3]) : "r"(a + UM_BLOCK_M * 128));
                            } else {
                                ll[0] = ll[1] = ll[2] = ll[3] = 0u;
                            }
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float2 rh = um_h2f(hh[j]), rl = um_h2f(ll[j]);
                                v[g * 8 + 2 * j] += rh.x + rl.x;
                                v[g * 8 + 2 * j + 1] += rh.y + rl.y;
                            }
                        }
                    }
                    if (e.act == SNNB_ACT_RELU) { // the common cases one instruction per element (the epilogue is issue-bound on short-K layers)
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.0f);
                    } else if (e.act == SNNB_ACT_NONE) {
                    } else if (e.act == SNNB_ACT_RELU6) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = fminf(fmaxf(v[j], 0.0f), 6.0f);
                    } else if (fast_act) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = fminf(fmaxf(v[j], v[j] * slope), hi_clip);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = (oc0 + c + j < e.OC) ? umma_act(v[j], e.act, e.alpha) : 0.0f; // out-of-line call
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) um_split2(v[2 * j], v[2 * j + 1], oh[kk][j], ol[kk][j]);
                }
            }
            if (k0 + 2 >= MAXC) { // the slab's last chunk pair is in registers
                EPI_STAMP(1);     // phase 1 done
                if (e.has_res && !res_ready) mbar_wait(e.res_bar, res_phase); // warps without a chunk in this slab still consume the phase
                if (e.has_res) res_phase ^= 1u;
                if (sl == nslabs - 1 && !e.part_src) { // last tcgen05.ld of the tile issued: the accumulator buffer may be reused
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(e.tmem_empty);
                }
            }
            // ---- staging buffer. The previous slab's / tile's bulk store has had the whole first chunk pair (and usually the
            // wait for the next accumulator) to finish READING the buffer; only now does anyone wait for it. ----
            if (k0 == 0) {
                if (!e.has_res) {
                    if (leader) {
                        if (elect_one()) {
                            if (e.two_stagings) bulk_wait_read1();
                            else bulk_wait_read0();
                        }
                        __syncwarp();
                    }
                    EPI_STAMP(2); // leader's wait for the previous store's reads
                    named_bar_sync(e.bar_id, NWARPS * 32);
                }
                EPI_STAMP(3); // bar A
            }
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const int k = k0 + kk, ci = NWARPS == 8 ? half + 2 * k : k;
                if (ci < (w >> 4)) {
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const uint32_t a = srow + ((((uint32_t) (ci * 2 + g)) ^ xr) << 4);
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(oh[kk][4 * g]), "r"(oh[kk][4 * g + 1]), "r"(oh[kk][4 * g + 2]), "r"(oh[kk][4 * g + 3])
                                     : "memory");
                        if (e.has_lo)
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + UM_BLOCK_M * 128), "r"(ol[kk][4 * g]), "r"(ol[kk][4 * g + 1]), "r"(ol[kk][4 * g + 2]),
                                         "r"(ol[kk][4 * g + 3])
                                         : "memory");
                    }
                }
            }
        }
        EPI_STAMP(4); // STS issued
        fence_async_smem();                 // generic-proxy smem writes -> visible to the TMA (async proxy)
        EPI_STAMP(5); // fence
        named_bar_sync(e.bar_id, NWARPS * 32);
        EPI_STAMP(6); // bar B
        if (leader) {
            if (!e.no_store && elect_one()) {
                tma_store_4d(sw ? e.o_hi64 : e.o_hiT, e.stg, slab_oc, c1, c2, c3);
                if (e.has_lo) tma_store_4d(sw ? e.o_lo64 : e.o_loT, e.stg + UM_BLOCK_M * 128, slab_oc, c1, c2, c3);
                bulk_commit();
            }
            __syncwarp();
        }
        EPI_STAMP(7); // store issued
    }
#undef EPI_STAMP
}
// Split-K: write this work item's raw fp32 accumulator tile (both column blocks added) to global memory, laid out
// [16-column chunk][float4 index][row][4 floats] so that every warp access is 512 contiguous bytes.
template <int NWARPS, int TERMS>
__device__ __forceinline__ void epilogue_dump_partial(const EpiArgs& e, uint32_t taddr, float* dst, int row, int half, int lane) {
    for (int c = (NWARPS == 8 ? half : 0) * 16; c < e.n_blk; c += (NWARPS == 8 ? 32 : 16)) {
        uint32_t r[16], r2[16];
        tmem_ld16(taddr + (uint32_t) c, r);
        if (TERMS == 3) {
            tmem_ld16(taddr + (uint32_t) (e.n_blk + c), r2);
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) r2[j] = 0u;
        }
        tmem_ld_wait();
        float4* d = reinterpret_cast<float4*>(dst) + (size_t) (c >> 4) * 4 * UM_BLOCK_M + row; // [chunk][j4][row][4 floats]
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4)
            d[j4 * UM_BLOCK_M] = make_float4(__uint_as_float(r[4 * j4]) + __uint_as_float(r2[4 * j4]), __uint_as_float(r[4 * j4 + 1]) + __uint_as_float(r2[4 * j4 + 1]),
                                __uint_as_float(r[4 * j4 + 2]) + __uint_as_float(r2[4 * j4 + 2]), __uint_as_float(r[4 * j4 + 3]) + __uint_as_float(r2[4 * j4 + 3]));
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(e.tmem_empty);
}

// After the last tile: the leader's bulk stores must have completed before the CTA (and its shared memory) goes away.
__device__ __forceinline__ void epilogue_drain(bool leader) {
    if (leader) {
        if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The kernel
// ---------------------------------------------------------------------------------------------------------------
// One work item of conv_umma_kernel: which tile, which K blocks, and - when the tile's K range is shared between CTAs - which piece
// of how many, plus the slot of its partial tiles.
struct WorkItem {
    int tile, kb0, kb1, piece, pieces, slot;
};
template <bool SK> // compile-time: the stream-K arithmetic (64-bit divisions) stays out of every other instantiation's issue loops
__host__ __device__ __forceinline__ WorkItem decode_work(const UmmaParams& p, int work, int total_tiles, int num_kb) {
    WorkItem w;
    if constexpr (!SK) {
        const int split = work / total_tiles;
        w.tile = work - split * total_tiles, w.kb0 = split * p.kb_per_split, w.kb1 = w.kb0 + p.kb_per_split < num_kb ? w.kb0 + p.kb_per_split : num_kb;
        w.piece = split, w.pieces = p.ksplit, w.slot = w.tile;
    } else if (work < p.sk_dp) {
        w.tile = work, w.kb0 = 0, w.kb1 = num_kb, w.piece = 0, w.pieces = 1, w.slot = 0;
    } else {
        const int c = (work - p.sk_dp) >> 2, j = (work - p.sk_dp) & 3;
        const long long b0 = (long long) c * p.sk_units / p.sk_ctas, b1 = (long long) (c + 1) * p.sk_units / p.sk_ctas; // this CTA's units
        const int jt = (int) (b0 / num_kb) + j; // tile (counted from sk_dp) of the CTA's j-th piece
        const long long t0 = (long long) jt * num_kb, t1 = t0 + num_kb;
        w.tile = p.sk_dp + jt, w.slot = jt;
        w.kb0 = (int) ((b0 > t0 ? b0 : t0) - t0), w.kb1 = (int) ((b1 < t1 ? b1 : t1) - t0);
        // CTA holding unit u: ((u + 1) * ctas - 1) / units
        const int c_first = (int) (((t0 + 1) * p.sk_ctas - 1) / p.sk_units), c_last = (int) ((t1 * p.sk_ctas - 1) / p.sk_units);
        w.piece = c - c_first, w.pieces = c_last - c_first + 1;
    }
    return w;
}
// Static schedule of a stream-K launch: CTA `cta` first works off the pieces of its K-block range, then its whole tiles cta, cta + grid, ...
// (pieces first: a cut tile's last arriver sums the partials while the other CTAs are busy with whole tiles, not at the very end of the
// launch with everybody waiting). Returns the work id after `work` (`end` when there is none) / the first one.
__host__ __device__ __forceinline__ int sk_next_work(const UmmaParams& p, int work, int cta, int grid, int num_kb, int end) {
    if (work < p.sk_dp) return work + grid < p.sk_dp ? work + grid : end;
    const int c = (work - p.sk_dp) >> 2, j = ((work - p.sk_dp) & 3) + 1;
    const long long b0 = (long long) c * p.sk_units / p.sk_ctas, b1 = (long long) (c + 1) * p.sk_units / p.sk_ctas;
    if (j < 4 && b0 / num_kb + j <= (b1 - 1) / num_kb) return work + 1;
    return cta < p.sk_dp ? cta : end;
}
__host__ __device__ __forceinline__ int sk_first_work(const UmmaParams& p, int cta, int end) {
    return cta < p.sk_ctas ? p.sk_dp + 4 * cta : (cta < p.sk_dp ? cta : end);
}

// K block kb of a plain-mode launch: the k x k taps of the input come first, (tap, 64-channel block) in order kb = tap * cblocks + cb;
// the sc_cblocks blocks of a folded shortcut follow. `wcol` is the block's first column in the packed weights.
struct KBlock {
    int sc, tap, cb, wcol;
};
__host__ __device__ __forceinline__ KBlock decode_kblock(const UmmaParams& p, int kb) {
    const int kb_main = p.ksize * p.ksize * p.cblocks;
    KBlock k;
    k.sc  = kb >= kb_main;
    k.tap = k.sc ? 0 : kb / p.cblocks;
    k.cb  = k.sc ? kb - kb_main : kb - k.tap * p.cblocks;
    k.wcol = (k.sc ? p.ksize * p.ksize : k.tap) * p.ICp + k.cb * UM_BLOCK_K;
    return k;
}
// The producer's walk over K blocks [kb0, kb1): decoded once, then stepped (no divisions per K block). f(kb, sc, cb, kx, ky, wcol).
// A range may straddle the end of the taps (split-K / stream-K pieces); the walk then switches to the shortcut operand once.
template <class F> __host__ __device__ __forceinline__ void for_each_kblock(const UmmaParams& p, int kb0, int kb1, F&& f) {
    const int ks = p.ksize, cbs = p.cblocks, icp = p.ICp, kb_main = ks * ks * cbs;
    const KBlock k0 = decode_kblock(p, kb0);
    int cb = k0.cb, kx = k0.tap % ks, ky = k0.tap / ks;
    int wk = k0.wcol - k0.cb * UM_BLOCK_K; // tap * ICp; past the taps: ks * ks * ICp, the shortcut's first column
    int kb = kb0;
    for (const int e = kb1 < kb_main ? kb1 : kb_main; kb < e; ++kb) {
        f(kb, false, cb, kx, ky, wk + cb * UM_BLOCK_K);
        if (++cb == cbs) {
            cb = 0, wk += icp;
            if (++kx == ks) kx = 0, ++ky;
        }
    }
    for (; kb < kb1; ++kb, ++cb) f(kb, true, cb, 0, 0, wk + cb * UM_BLOCK_K);
}

#define UM_TRACE(role, idx)                                                                          \
    do {                                                                                             \
        if (p.trace && blockIdx.x == 0 && lane == 0 && (idx) < 256) p.trace[(role) * 256 + (idx)] = clock64(); \
    } while (0)

// STAGES: depth of the operand ring. SPLIT_EPI: the eight epilogue warps work as TWO independent groups of four, group g
// owning accumulator buffer g (tiles alternate between the buffers) with its own staging buffer, named barrier, residual
// barrier and bulk-store queue, so one group's barrier / TMA-store latencies overlap the other group's arithmetic. Used for
// layers with a short K loop (1x1 convolutions), which run at the speed of the epilogue; pays for the second staging buffer
// with one ring stage (2 instead of 3).
// TERMS: how the fp32-faithful product is formed. 3 = A_hi x [B_hi ; B_lo] + A_lo x B_hi (fp16 weight pair, accumulator of two
// column blocks, n_blk <= 128); 2 = (A_hi + A_lo) x B16 with ONE fp16 weight plane (one column block, n_blk <= 256);
// 1 = A_hi x B_hi only (fp16 storage mode: no lo planes anywhere).
template <int STAGES, bool SPLIT_EPI, int TERMS, bool HALO, bool SK = false> // SK: stream-K work decomposition (UmmaParams::sk)
__global__ void __launch_bounds__(UM_THREADS, 1)
conv_umma_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo, const __grid_constant__ CUtensorMap tmB_hi,
                 const __grid_constant__ CUtensorMap tmB_lo, const __grid_constant__ CUtensorMap tmO_hi64, const __grid_constant__ CUtensorMap tmO_lo64,
                 const __grid_constant__ CUtensorMap tmO_hiT, const __grid_constant__ CUtensorMap tmO_loT, const __grid_constant__ CUtensorMap tmR_hi64,
                 const __grid_constant__ CUtensorMap tmR_lo64, const __grid_constant__ CUtensorMap tmR_hiT, const __grid_constant__ CUtensorMap tmR_loT,
                 const __grid_constant__ CUtensorMap tmS_hi, const __grid_constant__ CUtensorMap tmS_lo, const UmmaParams p) {
    extern __shared__ uint8_t smem_raw[];
    constexpr bool ONE_BLOCK = TERMS != 3 || SPLIT_EPI; // the accumulator is one column block of n_blk (else [hi.hi + lo.hi | hi.lo])
    constexpr int EPI_TERMS  = ONE_BLOCK ? 2 : 3;       // what the epilogue templates need to know: one block or two
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u; // SWIZZLE_128B tiles need 1024-byte alignment
    // HALO: [A ring: HL_A_STAGES x (hi plane, lo plane)] [B ring: STAGES x 32 KB] [staging]; else [ring: STAGES x 64 KB] [staging]
    const uint32_t b_ring    = smem_base + (HALO ? HL_A_STAGES * HL_A_STAGE_BYTES : 0);
    const uint32_t stg       = HALO ? b_ring + HL_B_RING_BYTES : smem_base + STAGES * UM_STAGE_BYTES; // epilogue staging (1024-aligned), one buffer per epilogue group
    const uint32_t bar_base  = stg + (SPLIT_EPI ? 2 : 1) * UM_STG_BYTES;
    // barrier slots (8 bytes each): full[0..S), empty[S..2S), tmem_full[2S..2S+2), tmem_empty[2S+2..2S+4), TMEM base slot, residual barrier
    auto full_bar       = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar      = [&](int s) { return bar_base + 8u * (STAGES + s); };
    auto tmem_full_bar  = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
    auto tmem_empty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
    const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
    const uint32_t res_bar   = bar_base + 8u * (2 * STAGES + 5); // SPLIT_EPI: group 1 uses the slot after the split-K flag (+16)
    // Dynamic work distribution. CTA b starts with work item b; every further item is drawn from a global counter by the
    // producer warp (persistent CTAs on a statically striped grid finished up to 17 % apart on store-heavy layers) and handed
    // to the MMA thread and the epilogue warps through this ring: id in sched_id[slot], full/empty mbarriers per slot.
    const uint32_t sched_base = bar_base + 8u * (2 * STAGES + 8); // behind the slots above (2 * STAGES + 8 of them)
    auto sched_full  = [&](int s) { return sched_base + 8u * s; };
    auto sched_empty = [&](int s) { return sched_base + 64u + 8u * s; };
    auto sched_id    = [&](int s) { return sched_base + 128u + 4u * s; };
    auto a_full_bar  = [&](int s) { return sched_base + 160u + 8u * s; }; // HALO: the halo-tile ring
    auto a_empty_bar = [&](int s) { return sched_base + 176u + 8u * s; };
    // consumer side: wait for sequence number `seq`, read its work id, release the slot (one arrive per consuming warp)
    auto sched_take = [&](int seq, bool arrive) {
        const int slot = seq & (UM_SCHED_SLOTS - 1);
        mbar_wait(sched_full(slot), (uint32_t) (seq / UM_SCHED_SLOTS) & 1u);
        int w;
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(sched_id(slot)) : "memory");
        if (arrive) mbar_arrive(sched_empty(slot));
        return w;
    };

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger(); // the next kernel may start launching; it waits for this grid's completion before touching memory
    if (warp == 0 && lane == 0) {
        mbar_init(res_bar, 1);
        mbar_init(res_bar + 16u, 1);
        tma_prefetch_desc(&tmO_hi64);
        tma_prefetch_desc(&tmO_lo64);
        tma_prefetch_desc(&tmA_hi);
        tma_prefetch_desc(&tmA_lo);
        tma_prefetch_desc(&tmB_hi);
        tma_prefetch_desc(&tmB_lo);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        if (HALO)
            for (int s = 0; s < HL_A_STAGES; ++s) {
                mbar_init(a_full_bar(s), 1);
                mbar_init(a_empty_bar(s), 1);
            }
        for (int s = 0; s < UM_SCHED_SLOTS; ++s) {
            mbar_init(sched_full(s), 1);
            mbar_init(sched_empty(s), 1 + UM_EPI_WARPS); // the MMA thread + one lane of every epilogue warp
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tmem_full_bar(a), 1);
            mbar_init(tmem_empty_bar(a), SPLIT_EPI ? UM_EPI_WARPS / 2 : UM_EPI_WARPS); // one arrive per epilogue warp that drains the buffer
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, UM_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    // The WEIGHTS of this CTA's first work item do not depend on the previous kernel: their loads go out before the dependency wait
    // (plain mode: the first K block's; halo mode: the first three taps'), so only the activations' latency is left after it.
    const int pre_total_tiles = p.tiles_x * p.tiles_y * p.tiles_n * p.tiles_oc;
    const int pre_num_kb      = p.ksize * p.ksize * p.cblocks + p.sc_cblocks;
    const int pre_end         = SK ? p.sk_dp + 4 * p.sk_ctas : pre_total_tiles * p.ksplit; // one past the last work id
    const int first_work      = SK ? sk_first_work(p, (int) blockIdx.x, pre_end) : (int) blockIdx.x;
    const bool pre_b          = (p.ablate & (2 | 16)) == 0 && first_work < pre_end; // ablate 16: no early weight loads (results stay correct)
    if (warp == 0 && pre_b && elect_one()) {
        const WorkItem w0 = decode_work<SK>(p, first_work, pre_total_tiles, pre_num_kb);
        const int tile    = w0.tile;
        const int oc0  = (tile / (p.tiles_x * p.tiles_y * p.tiles_n)) * p.n_blk;
        const uint32_t b_lo_off = (uint32_t) p.n_blk * 128u;
        if (HALO) {
            for (int tap = 0; tap < 3; ++tap) {
                const uint32_t sB = b_ring + tap * p.b_stage_bytes, fb = full_bar(tap);
                mbar_expect_tx(fb, (TERMS == 3 ? 2u : 1u) * (uint32_t) p.n_blk * 128u);
                tma_load_2d(sB, &tmB_hi, fb, tap * p.ICp, oc0);
                if (TERMS == 3) tma_load_2d(sB + b_lo_off, &tmB_lo, fb, tap * p.ICp, oc0);
            }
        } else {
            const int wcol    = decode_kblock(p, w0.kb0).wcol;
            const uint32_t fb = full_bar(0);
            mbar_expect_tx(fb, (TERMS == 1 ? 1u : 2u) * (uint32_t) p.rows_used * 128u + (TERMS == 3 ? 2u : 1u) * (uint32_t) p.n_blk * 128u);
            tma_load_2d(smem_base + 2 * UM_A_BYTES, &tmB_hi, fb, wcol, oc0);
            if (TERMS == 3) tma_load_2d(smem_base + 2 * UM_A_BYTES + b_lo_off, &tmB_lo, fb, wcol, oc0);
        }
    }
    // everything above (barriers, TMEM, tensor-map prefetch, first weights) overlapped with the previous kernel's tail. A folded
    // shortcut's operand was written two launches back, not by the previous grid: that grid itself passed this wait on ITS
    // predecessor before it could complete, so once it has completed every earlier grid has too.
    pdl_wait();
    if (warp == 0) UM_TRACE(5, 0); // kernel entry (after the dependency wait)
    if (p.trace && threadIdx.x == 0) { // wall-clock (ns) envelope over ALL CTAs: [5][8] = earliest entry, [5][9] = latest exit, [5][10..11] CTA 0's own
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        atomicMin(reinterpret_cast<unsigned long long*>(p.trace) + 5 * 256 + 8, g);
        if (blockIdx.x == 0) p.trace[5 * 256 + 10] = (long long) g;
    }

    if (warp == 0) UM_TRACE(5, 1); // setup done

    const int m_tiles     = p.tiles_x * p.tiles_y * p.tiles_n;
    const int total_tiles = m_tiles * p.tiles_oc;
    const int num_kb      = p.ksize * p.ksize * p.cblocks + p.sc_cblocks;
    const int total_work  = SK ? p.sk_dp + 4 * p.sk_ctas : total_tiles * p.ksplit; // work item = (tile, K range); one past the last work id

    if (warp == 0) {
        // ===================== TMA producer =====================
        {
            int stage = 0, hstage = 0;
            uint32_t phase = 0, hphase = 0;
            (void) hstage, (void) hphase;
            const uint32_t tx_bytes = (TERMS == 1 ? 1u : 2u) * (uint32_t) p.rows_used * 128u + (TERMS == 3 ? 2u : 1u) * (uint32_t) p.n_blk * 128u;
            const int cbs = p.cblocks, icp = p.ICp;
            const bool skip_tma = (p.ablate & 2) != 0;
            const uint32_t b_lo_off = (uint32_t) p.n_blk * 128u; // B_lo rows follow B_hi's: one [2 n_blk x 64] operand
            int tr = 0;
            const int draws_total = max(0, total_work - (int) gridDim.x) + (int) gridDim.x; // every CTA's last draw is past the end
            int work = first_work;
            for (int seq = 0;; ++seq) {
                if (p.ablate & 32) producer_progress(lane, ((unsigned) seq << 16) | 0x01u); // SNNB_UMMA_ABLATE=32: leave a trail for the time-out report
                {   // publish this sequence number's work id
                    const int slot = seq & (UM_SCHED_SLOTS - 1);
                    mbar_wait(sched_empty(slot), ((uint32_t) (seq / UM_SCHED_SLOTS) & 1u) ^ 1u);
                    if (elect_one()) {
                        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sched_id(slot)), "r"(work) : "memory");
                        mbar_arrive(sched_full(slot));
                    }
                }
                if (p.ablate & 32) producer_progress(lane, ((unsigned) seq << 16) | 0x02u);
                if (work >= total_work) break;
                // The next work item is drawn NOW but its result is not touched until this item's loads are issued: 148 CTAs hit the same
                // counter at kernel start (a ~1.3 k clk round trip). r01 tested the result right away (`if (c == last) reset`), which put that
                // round trip in front of every item's first load - the producer's whole run-ahead margin (r02 trace: first load 2.3-5.4 k clk
                // after kernel entry, ~1.3 k clk of bubble at every tile boundary).
                int drawn = 0;
                if (!SK && elect_one()) drawn = atomicAdd(p.sched_counter, 1);
                auto take_next = [&]() { // consumes the draw: next work id for all lanes; the launch's last draw re-zeroes the counter
                    if constexpr (SK) return sk_next_work(p, work, (int) blockIdx.x, (int) gridDim.x, num_kb, total_work); // static schedule
                    const int c = __shfl_sync(0xffffffffu, drawn, 0); // elect.sync picks lane 0 of the converged warp
                    if (lane == 0 && c == draws_total - 1) *p.sched_counter = 0;
                    return (int) gridDim.x + c;
                };
                const WorkItem wi = decode_work<SK>(p, work, total_tiles, num_kb);
                const int tile = wi.tile;
                const int m_idx = tile % m_tiles, oc_idx = tile / m_tiles;
                const int bx = m_idx % p.tiles_x, by = (m_idx / p.tiles_x) % p.tiles_y, bn = m_idx / (p.tiles_x * p.tiles_y);
                const int ix0 = bx * p.tw * p.stride - p.pad_x, iy0 = by * p.th * p.stride - p.pad_y, n0 = bn * p.tn;
                const int oc0 = oc_idx * p.n_blk;
                const int kb0 = wi.kb0, kb1 = wi.kb1;
                // Keep this loop lean: it runs once per K block and every stall here delays the whole pipeline (no divisions,
                // no parameter loads: ncu r01 showed ~60 dependent scalar instructions/iteration bounding the kernel).
                // K block kb = (ky * ks + kx) * cbs + cb, then a folded shortcut's blocks; the counters are decoded once per work item
                // and then stepped (for_each_kblock).
                if constexpr (HALO) {
                    // K order (cb, tap): one halo tile per channel block, then the nine taps' weights. The halo tile of the NEXT
                    // unit (next channel block, or the next work item's first) is requested one unit ahead, after this unit's first
                    // weight stages are in flight: its ~1 us latency used to sit exposed at every tile boundary (r02 trace: ~2 k clk
                    // of 7.5 k per 56x56x64 tile).
                    auto issue_halo = [&](int w, int cb) {
                        const int tile_ = w % total_tiles, m_ = tile_ % m_tiles;
                        const int bx_ = m_ % p.tiles_x, by_ = (m_ / p.tiles_x) % p.tiles_y, bn_ = m_ / (p.tiles_x * p.tiles_y);
                        mbar_wait(a_empty_bar(hstage), hphase ^ 1u);
                        if (elect_one()) {
                            const uint32_t sA = smem_base + hstage * HL_A_STAGE_BYTES, fb = a_full_bar(hstage);
                            if (skip_tma) {
                                mbar_arrive(fb);
                            } else {
                                mbar_expect_tx(fb, (TERMS == 1 ? 1u : 2u) * (uint32_t) (HL_W * HL_H * 128));
                                tma_load_4d(sA, &tmA_hi, fb, cb * UM_BLOCK_K, bx_ * HL_TW - p.pad_x, by_ * HL_TH - p.pad_y, bn_);
                                if (TERMS >= 2) tma_load_4d(sA + HL_PLANE, &tmA_lo, fb, cb * UM_BLOCK_K, bx_ * HL_TW - p.pad_x, by_ * HL_TH - p.pad_y, bn_);
                            }
                        }
                        __syncwarp();
                        if (++hstage == HL_A_STAGES) hstage = 0, hphase ^= 1u;
                    };
                    if (seq == 0) issue_halo(work, 0); // prologue: every later unit's tile is requested by its predecessor
                    int nwork = total_work;           // next work item, known once the atomic draw above has returned
                    for (int cb = 0; cb < cbs; ++cb) {
                        int wk = cb * UM_BLOCK_K;
                        for (int tap = 0; tap < 9; ++tap, wk += icp) {
                            if (tap == 3) { // three weight stages are in flight: now the next unit's halo tile
                                if (cb + 1 < cbs) {
                                    issue_halo(work, cb + 1);
                                } else {
                                    nwork = take_next();
                                    if (nwork < total_work) issue_halo(nwork, 0);
                                }
                            }
                            // This CTA's first three weight stages went out before the dependency wait. They must not be waited for either:
                            // the MMA thread may already have consumed such a stage and committed its empty barrier, and a wait for
                            // "the phase before the first" would then block for ever (seen as a rare hang of the first launches, when
                            // the producer was slow to get here: cold instruction cache).
                            const bool pre_stage = seq == 0 && cb == 0 && tap < 3 && pre_b;
                            if (!pre_stage) mbar_wait(empty_bar(stage), phase ^ 1u);
                            UM_TRACE(0, tr);
                            ++tr;
                            if (pre_stage) {
                            } else if (elect_one()) {
                                const uint32_t sB = b_ring + stage * p.b_stage_bytes, fb = full_bar(stage);
                                if (skip_tma) {
                                    mbar_arrive(fb);
                                } else {
                                    mbar_expect_tx(fb, (TERMS == 3 ? 2u : 1u) * (uint32_t) p.n_blk * 128u);
                                    tma_load_2d(sB, &tmB_hi, fb, wk, oc0);
                                    if (TERMS == 3) tma_load_2d(sB + b_lo_off, &tmB_lo, fb, wk, oc0);
                                }
                            }
                            if (++stage == p.b_stages) stage = 0, phase ^= 1u;
                        }
                    }
                    work = nwork;
                    continue;
                }
                // the folded shortcut's box: the same output pixels at its own stride, pad 0 (a 1x1 convolution)
                const int sx0 = bx * p.tw * p.sc_stride, sy0 = by * p.th * p.sc_stride;
                for_each_kblock(p, kb0, kb1, [&](int kb, bool sc, int cb, int kx, int ky, int wcol) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    UM_TRACE(0, tr);
                    ++tr;
                    if (elect_one()) {
                        const uint32_t sA = smem_base + stage * UM_STAGE_BYTES, fb = full_bar(stage);
                        if (skip_tma) {
                            mbar_arrive(fb);
                        } else {
                            const bool pre = seq == 0 && kb == kb0 && pre_b; // expect_tx + the weights went out before the dependency wait
                            if (!pre) mbar_expect_tx(fb, tx_bytes);
                            const CUtensorMap* a_hi = sc ? &tmS_hi : &tmA_hi;
                            const CUtensorMap* a_lo = sc ? &tmS_lo : &tmA_lo;
                            const int ax = sc ? sx0 : ix0 + kx, ay = sc ? sy0 : iy0 + ky;
                            tma_load_4d(sA, a_hi, fb, cb * UM_BLOCK_K, ax, ay, n0);
                            if (TERMS >= 2) tma_load_4d(sA + UM_A_BYTES, a_lo, fb, cb * UM_BLOCK_K, ax, ay, n0);
                            if (!pre) {
                                tma_load_2d(sA + 2 * UM_A_BYTES, &tmB_hi, fb, wcol, oc0);
                                if (TERMS == 3) tma_load_2d(sA + 2 * UM_A_BYTES + b_lo_off, &tmB_lo, fb, wcol, oc0);
                            }
                        }
                    }
                    if (++stage == STAGES) stage = 0, phase ^= 1u;
                });
                work = take_next();
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int stage = 0;
        uint32_t phase = 0;
        // 3-term split product with TWO MMAs per K step: A_hi x [B_hi ; B_lo] (N = 2 n_blk, two column blocks) and
        // A_lo x B_hi (N = n_blk, onto the first block); the epilogue adds the blocks. Same math as three N = n_blk MMAs, but
        // A_hi is fetched from shared memory once instead of twice and there are 8 instead of 12 issues per K block.
        const uint32_t idesc_cat = TERMS == 3 ? make_idesc(UM_BLOCK_M, 2 * p.n_blk) : 0u;
        const uint32_t idesc     = make_idesc(UM_BLOCK_M, p.n_blk);
        // Descriptor of stage 0's A_hi tile; every other operand is this plus a constant in the 16-byte address field (all of
        // shared memory is < 256 KB, so the 14-bit field never carries). Keeps the per-K-block preamble to a couple of adds:
        // the issue of tcgen05.mma does not run ahead of the tensor pipe, so every scalar clock here is a lost MMA clock.
        const uint64_t desc0 = make_smem_desc(smem_base);
        // ONE thread runs the whole issue loop. Issuing tcgen05.mma stalls the thread while the tensor pipe's short queue is
        // full, so scalar work placed BETWEEN the MMAs of a K block overlaps with them, while work between K blocks is lost
        // tensor time: the look-ahead test of the next stage's barrier and the bookkeeping sit before the last two MMAs.
        if (elect_one()) {
            int it = 0, tr = 0, hstage = 0;
            uint32_t hphase = 0;
            (void) hstage, (void) hphase;
            bool ready = false; // full_bar(stage) already observed complete by the look-ahead
            const bool no_mma = (p.ablate & 4) != 0;
            for (;; ++it) {
                const int work = sched_take(it, true);
                if (work >= total_work) break;
                const int acc = it & 1;
                const uint32_t acc_phase = (uint32_t) (it >> 1) & 1u;
                mbar_wait(tmem_empty_bar(acc), acc_phase ^ 1u); // epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t) (acc * UM_ACC_COLS);
                if constexpr (HALO) {
                    const uint64_t bdesc0 = make_smem_desc(b_ring);
                    for (int cb = 0; cb < p.cblocks; ++cb) {
                        mbar_wait(a_full_bar(hstage), hphase); // this channel block's halo tile has landed
                        // SBO = the halo's row pitch (10 pixels): 8-row group g of tap (ky,kx) starts (g + ky) * 10 + kx pixels into the tile
                        const uint64_t halo = make_smem_desc_sbo(smem_base + hstage * HL_A_STAGE_BYTES, HL_W * 128);
                        int tap_off = 0; // (ky * HL_W + kx) * 128 B, in 16-byte units
                        for (int tap = 0; tap < 9; ++tap) {
                            if (!ready) mbar_wait(full_bar(stage), phase); // this tap's weights have landed
                            tc_fence_after();
                            UM_TRACE(1, tr);
                            const uint64_t a_hi = halo + (uint64_t) (uint32_t) tap_off, a_lo = a_hi + (HL_PLANE >> 4);
                            const uint64_t b_cat = bdesc0 + (uint64_t) (uint32_t) (stage * (p.b_stage_bytes >> 4));
                            const uint32_t first = (cb > 0 || tap > 0) ? 1u : 0u;
                            // First K step, then the look-ahead test of the next stage's barrier (its ~150 clk latency hides behind
                            // the six MMAs still to be issued: behind only two, as in r01, the pipe ran dry ~180 clk per K block),
                            // then the rest.
                            if (!no_mma) {
                                umma_f16(d_tmem, a_hi, b_cat, TERMS == 3 ? idesc_cat : idesc, first);
                                if (TERMS == 2) umma_f16(d_tmem, a_lo, b_cat, idesc, 1u);
                            }
                            const int cur         = stage;
                            const uint32_t nphase = phase ^ (stage == p.b_stages - 1 ? 1u : 0u);
                            stage                 = stage == p.b_stages - 1 ? 0 : stage + 1;
                            phase                 = nphase;
                            ready                 = mbar_test_wait(full_bar(stage), phase); // non-blocking look-ahead
                            if (!no_mma) {
                                if (TERMS == 3) {
#pragma unroll
                                    for (int j = 1; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc_cat, 1u);
#pragma unroll
                                    for (int j = 0; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_lo + 2u * j, b_cat + 2u * j, idesc, 1u);
                                } else if (TERMS == 2) {
#pragma unroll
                                    for (int j = 1; j < UM_BLOCK_K / 16; ++j) {
                                        umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc, 1u);
                                        umma_f16(d_tmem, a_lo + 2u * j, b_cat + 2u * j, idesc, 1u);
                                    }
                                } else {
#pragma unroll
                                    for (int j = 1; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc, 1u);
                                }
                            }
                            umma_commit(empty_bar(cur)); // weight slot free once these MMAs retire
                            UM_TRACE(2, tr);
                            ++tr;
                            tap_off += (tap % 3 == 2) ? ((HL_W - 2) * 128 >> 4) : (128 >> 4); // next tap: +1 pixel, or to the next halo row
                        }
                        umma_commit(a_empty_bar(hstage)); // halo tile free once all nine taps have retired
                        if (++hstage == HL_A_STAGES) hstage = 0, hphase ^= 1u;
                    }
                    umma_commit(tmem_full_bar(acc)); // accumulator complete -> epilogue
                    continue;
                }
                const WorkItem wi = decode_work<SK>(p, work, total_tiles, num_kb);
                const int kb0 = wi.kb0, kb1 = wi.kb1;
                for (int kb = kb0; kb < kb1; ++kb) {
                    if (!ready) mbar_wait(full_bar(stage), phase); // TMA bytes have landed
                    tc_fence_after();
                    UM_TRACE(1, tr);
                    const uint64_t a_hi = desc0 + (uint64_t) (uint32_t) (stage * (UM_STAGE_BYTES >> 4)), a_lo = a_hi + (UM_A_BYTES >> 4);
                    const uint64_t b_cat = a_hi + (2 * UM_A_BYTES >> 4); // rows [0, n_blk) = B_hi, [n_blk, 2 n_blk) = B_lo
                    // UMMA_K = 16 fp16 = 32 bytes: K step j advances the start address by 2 (x16 B)
                    const uint32_t first = kb > kb0 ? 1u : 0u;
                    // ONE_BLOCK (short-K layers, 3-term): all three products go to the SAME accumulator block as separate N = n_blk MMAs
                    // (12 instead of 8 per K block, A_hi fetched twice) - these layers run at the speed of their epilogue, not of the
                    // tensor pipe, and this way the epilogue reads one TMEM block instead of two and adds nothing.
                    const uint64_t b_lo = b_cat + (uint64_t) ((uint32_t) p.n_blk * 8u); // B_lo rows follow B_hi's (n_blk x 128 B)
                    // first K step | look-ahead test of the next stage (latency hidden behind the remaining MMAs) | the rest
                    if (!no_mma) {
                        umma_f16(d_tmem, a_hi, b_cat, (TERMS == 3 && !ONE_BLOCK) ? idesc_cat : idesc, first);
                        if (TERMS == 2) umma_f16(d_tmem, a_lo, b_cat, idesc, 1u);
                        if (TERMS == 3 && ONE_BLOCK) umma_f16(d_tmem, a_hi, b_lo, idesc, 1u);
                    }
                    const int cur         = stage;
                    const uint32_t nphase = phase ^ (stage == STAGES - 1 ? 1u : 0u);
                    stage                 = stage == STAGES - 1 ? 0 : stage + 1;
                    phase                 = nphase;
                    ready                 = mbar_test_wait(full_bar(stage), phase); // non-blocking
                    if (!no_mma) {
                        if (TERMS == 3 && ONE_BLOCK) {
#pragma unroll
                            for (int j = 1; j < UM_BLOCK_K / 16; ++j) {
                                umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc, 1u);
                                umma_f16(d_tmem, a_hi + 2u * j, b_lo + 2u * j, idesc, 1u);
                            }
#pragma unroll
                            for (int j = 0; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_lo + 2u * j, b_cat + 2u * j, idesc, 1u);
                        } else if (TERMS == 3) {
#pragma unroll
                            for (int j = 1; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc_cat, 1u);
#pragma unroll
                            for (int j = 0; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_lo + 2u * j, b_cat + 2u * j, idesc, 1u);
                        } else if (TERMS == 2) {
#pragma unroll
                            for (int j = 1; j < UM_BLOCK_K / 16; ++j) {
                                umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc, 1u);
                                umma_f16(d_tmem, a_lo + 2u * j, b_cat + 2u * j, idesc, 1u);
                            }
                        } else {
#pragma unroll
                            for (int j = 1; j < UM_BLOCK_K / 16; ++j) umma_f16(d_tmem, a_hi + 2u * j, b_cat + 2u * j, idesc, 1u);
                        }
                    }
                    umma_commit(empty_bar(cur));                           // smem slot free once these MMAs retire
                    if (kb == kb1 - 1) umma_commit(tmem_full_bar(acc)); // accumulator complete -> epilogue
                    UM_TRACE(2, tr);
                    ++tr;
                }
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue (8 warps): see epilogue_tile =====================
        const int q    = warp & 3;        // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2; // which interleaved set of 16-column chunks this warp owns
        const int row  = q * 32 + lane;
        EpiArgs e;
        e.o_hi64 = &tmO_hi64, e.o_lo64 = &tmO_lo64, e.o_hiT = &tmO_hiT, e.o_loT = &tmO_loT;
        e.r_hi64 = &tmR_hi64, e.r_lo64 = &tmR_lo64, e.r_hiT = &tmR_hiT, e.r_loT = &tmR_loT;
        e.bias = p.bias, e.n_blk = p.n_blk, e.OC = p.OC, e.act = p.act, e.has_res = p.has_res, e.rows_box = p.rows_used, e.alpha = p.alpha;
        e.has_lo = p.has_lo;
        const int grp = SPLIT_EPI ? half : 0;                 // epilogue group of this warp
        const bool leader = warp == (SPLIT_EPI ? 2 + 4 * grp : 2); // the group's TMA-issuing warp
        e.stg = stg + grp * UM_STG_BYTES, e.res_bar = res_bar + 16u * grp, e.bar_id = 1 + grp;
        e.part_src = nullptr, e.part_splits = 0;
        const uint32_t last_flag = bar_base + 8u * (2 * STAGES + 6); // split-K: "this CTA arrived last" broadcast slot
        uint32_t res_phase = 0;
        int it = 0;
        for (;; ++it) {
            const int work = sched_take(it, lane == 0);
            if (work >= total_work) break;
            const WorkItem wi = decode_work<SK>(p, work, total_tiles, num_kb);
            const int tile = wi.tile;
            const int acc = it & 1;
            const uint32_t acc_phase = (uint32_t) (it >> 1) & 1u;
            if (SPLIT_EPI && acc != grp) continue; // the other group's accumulator buffer
            const int m_idx = tile % m_tiles, oc_idx = tile / m_tiles;
            const int bx = m_idx % p.tiles_x, by = (m_idx / p.tiles_x) % p.tiles_y, bn = m_idx / (p.tiles_x * p.tiles_y);
            if (p.has_res && wi.pieces == 1 && !(p.ablate & 1)) epilogue_residual_load(e, 0, oc_idx * p.n_blk, bx * p.tw, by * p.th, bn * p.tn, leader);
            mbar_wait(tmem_full_bar(acc), acc_phase);
            tc_fence_after();
            if (leader) UM_TRACE(3, it);
            e.tmem_empty = tmem_empty_bar(acc);
            e.trace = p.trace, e.trace_seq = it;
            const uint32_t taddr = tmem_base + ((uint32_t) (q * 32) << 16) + (uint32_t) (acc * UM_ACC_COLS);
            if (p.ablate & 1) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(e.tmem_empty);
                continue;
            }
            if (wi.pieces > 1) {
                float* tile_parts = p.partials + (size_t) wi.slot * (SK ? 4 : p.ksplit) * (UM_BLOCK_M * p.n_blk);
                epilogue_dump_partial<UM_EPI_WARPS, EPI_TERMS>(e, taddr, tile_parts + (size_t) wi.piece * (UM_BLOCK_M * p.n_blk), row, half, lane);
                __threadfence(); // partial tile visible device-wide before the arrival is counted
                named_bar_sync(1, UM_EPI_WARPS * 32);
                if (warp == 2 && lane == 0) {
                    const int old  = atomicAdd(p.counters + wi.slot, 1);
                    const int last = old == wi.pieces - 1;
                    if (last) p.counters[wi.slot] = 0; // every piece has arrived: leave the counter ready for the next launch
                    asm volatile("st.shared.b32 [%0], %1;" ::"r"(last_flag), "r"(last) : "memory");
                }
                named_bar_sync(1, UM_EPI_WARPS * 32);
                int last;
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(last) : "r"(last_flag) : "memory");
                if (!last) continue;
                __threadfence();
                e.part_src = tile_parts, e.part_splits = wi.pieces;
                if (p.has_res) epilogue_residual_load(e, 0, oc_idx * p.n_blk, bx * p.tw, by * p.th, bn * p.tn, leader);
            }
            if (SPLIT_EPI)
                epilogue_tile<UM_EPI_WARPS / 2, EPI_TERMS>(e, taddr, oc_idx * p.n_blk, bx * p.tw, by * p.th, bn * p.tn, row, 0, leader, lane, res_phase);
            else
                epilogue_tile<UM_EPI_WARPS, EPI_TERMS>(e, taddr, oc_idx * p.n_blk, bx * p.tw, by * p.th, bn * p.tn, row, half, leader, lane, res_phase);
            e.part_src = nullptr;
            if (leader) UM_TRACE(4, it);
        }
        epilogue_drain(leader);
    }

    if (warp == 0) UM_TRACE(5, 2); // producer done
    tc_fence_before();
    __syncthreads();
    if (warp == 0) UM_TRACE(5, 3); // all roles done
    if (p.trace && threadIdx.x == 0) {
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        atomicMax(reinterpret_cast<unsigned long long*>(p.trace) + 5 * 256 + 9, g);
        if (blockIdx.x == 0) p.trace[5 * 256 + 11] = (long long) g;
    }
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, UM_TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Small-input-channel convolution (IC <= 8: the 7x7 / 3x3 RGB stems, ESPCN's 1-channel 5x5) on the same tensor cores,
// with a ZERO-COPY sliding-window A operand.
//
// With C padded to 8 fp16 one pixel is ONE 16-byte vector per plane = exactly one K "chunk" of a tcgen05 K-major
// operand. In the un-swizzled (SWIZZLE_NONE) canonical layout row m / chunk c of A is read from
//        start + (m/8)*SBO + (m%8)*16 B + c*LBO,
// and nothing stops LBO from being 16 B: chunk c of row m is then simply pixel m + c of a dense pixel row in shared
// memory - the convolution's sliding window, expressed in the descriptor (probed on B200: tools/umma_desc_probe.cu).
// So for every filter row ky the producer TMA-loads ONE dense row segment per column parity (for stride 2 the even and
// odd input columns are de-interleaved by the tensor map's 32-byte pixel stride; out-of-image pixels are zero-filled =
// constant padding) and the MMA warp issues one K=16 step per pair of taps: no im2col, no producer warps, no copies.
// L2 -> SM traffic per 128-pixel tile: kh * s * ~136 * 16 B * 2 planes (61 KB for the 7x7 stem) instead of 224 KB of
// gathered 16-byte requests. The weight panel [kh][n_blk][64] (hi + lo, K columns in RowPlan order) is loaded once per
// persistent CTA and stays resident. Tiles = up to 128 consecutive output pixels of one output row.
//
// FEED mode (r02; stride 2, <= 4 input channels = the RGB stems): the input kernels also write a compact copy of the image with
// FOUR channels per pixel and zero margins (snnb_tensor::feed_hi). With 8-byte pixels one 16-byte K chunk is a PAIR of adjacent
// pixels, and for stride 2 the window of output pixel m starts at pixel 2 m = 16 m bytes: the plain dense row is already the
// canonical operand (row pitch 16 B, LBO 16 B) - no parity de-interleave, half the K (7 taps x 4 channels + 1 pad tap = 32 instead of
// 64), one contiguous bulk copy per plane and filter row, real zeros instead of out-of-bounds fill (FeedPlan, snnb_internal.h).
// ---------------------------------------------------------------------------------------------------------------
constexpr int RW_MAX_STAGES    = 16;                           // ring depth is chosen per launch: whatever shared memory is left, see RowWinParams::stages
constexpr int RW_EPI_WARPS     = 8;
constexpr int RW_THREADS       = 64 + 32 * RW_EPI_WARPS;
constexpr int RW_MAX_N         = 64;
constexpr int RW_BOXW          = 144;                          // 128 tile pixels + up to 8 of window overhang, padded
constexpr int RW_ARR_BYTES     = RW_BOXW * 16;                 // one (plane, parity) pixel row segment
constexpr int RW_SMEM_BYTES    = 227 * 1024;                   // everything: resident weight panels | epilogue staging | A ring | barriers
constexpr int RW_BAR_BYTES     = 512;
constexpr int RW_B_MAX_BYTES   = RW_SMEM_BYTES - 1024 - RW_BAR_BYTES - UM_STG_BYTES - 4 * 4 * RW_ARR_BYTES; // weights must leave room for >= 4 stages

struct RowWinParams {
    __half* out_hi;
    __half* out_lo;
    const float* bias;
    int N, OH, OW, OC, OCp, n_blk, ocr;
    int kh, stride, pad_y;
    int tiles_x;
    int parities, dmin[2];
    int ksteps, panels, ks_parity[8], ks_erel[8]; // panels = ceil(ksteps / 4) weight panels of 64 K columns per filter row
    int act;
    float alpha;
    long long* trace; // profiling aid, see UmmaParams
    int ablate;       // profiling aid (SNNB_UMMA_ABLATE, results WRONG when set): 1 skip the epilogue work, 2 the activation loads, 4 the MMAs, 8 the TMA stores
    // FEED mode (stride 2, <= 4 input channels; FeedPlan in snnb_internal.h): the A rows come from the input tensor's compact
    // 4-channel copy, one contiguous segment per plane and filter row (a plain bulk copy, the margins are real zeros)
    const __half* feed_hi;
    const __half* feed_lo;
    int feed_h, feed_w, feed_py;
    uint32_t feed_seg_bytes; // 0 = not in feed mode
    // shared-memory carve-up (host-computed): the weight panels take b_bytes (multiple of 1024), the ring gets `stages` stages of
    // stage_bytes = planes x parities x RW_ARR_BYTES; the lo plane's arrays follow the hi plane's at lo_off. The ring is as deep as
    // shared memory allows: a stage is only ~2-9 KB, and the cycle load -> MMA -> commit -> producer wake-up is ~2.5 k clk long, so a
    // 5-deep ring ran the 7x7 stem at one stage per ~560 clk whatever the stage's own work was (profiles/r02_stem_ablation.txt).
    int stages;
    uint32_t stage_bytes, lo_off, b_bytes;
    // FEED mode: a stage holds `rows_per_stage` filter rows (row_bytes each: hi segment, lo segment), released by ONE tcgen05.commit -
    // a commit costs the issuing thread ~52 clk and a stage boundary ~100 more, against 224 clk of MMAs per filter row of the 7x7 stem
    int rows_per_stage;
    uint32_t row_bytes;
    int stg_bufs; // epilogue staging buffers (2: alternate tiles, see EpiArgs::two_stagings)
    int feed_prows; // feed mode: 128-byte weight rows per output channel = ceil(kh / FeedPlan::rows_per_panel)
};

// SWIZZLE_NONE K-major descriptor with an overlapping K stride: LBO = 16 B (next chunk = next pixel), SBO = 128 B
// (8 rows x 16 B), version 1, layout type 0.
__device__ __forceinline__ uint64_t make_window_desc(uint32_t saddr) { return (uint64_t) ((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (8ull << 32) | (1ull << 46); }

// FKS > 0: FEED mode with FKS K steps per filter row (see RowWinParams::feed_hi). Its producer and MMA-issue loops are written out
// separately and kept to a few dozen instructions per stage: both run in ONE thread, a stage of the 7x7 stem holds only four MMAs
// (224 clk of tensor time), and the generic loops below cost ~290 SASS instructions = ~400 clk per stage whatever the stage's work
// was (profiles/r02_stem_ablation.txt: with loads, MMAs and epilogue all ablated the kernel still took 48 of its 75 us).
template <int TERMS, int FKS> // TERMS: see conv_umma_kernel
__global__ void __launch_bounds__(RW_THREADS, 1)
conv_rowwin_kernel(const __grid_constant__ CUtensorMap tmA_hi0, const __grid_constant__ CUtensorMap tmA_hi1, const __grid_constant__ CUtensorMap tmA_lo0,
                   const __grid_constant__ CUtensorMap tmA_lo1, const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                   const __grid_constant__ CUtensorMap tmO_hi, const __grid_constant__ CUtensorMap tmO_lo, const RowWinParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sB = smem_base; // weight panel: per kernel row ky, [n_blk rows of B_hi ; n_blk rows of B_lo] x 128 B
    const uint32_t stg      = smem_base + p.b_bytes; // epilogue staging (1024-aligned)
    const uint32_t sA0      = stg + (uint32_t) p.stg_bufs * UM_STG_BYTES;
    const uint32_t bar_base = sA0 + (uint32_t) p.stages * p.stage_bytes;
    const int RW_STAGES     = p.stages;
    auto full_bar       = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar      = [&](int s) { return bar_base + 8u * (RW_MAX_STAGES + s); };
    auto tmem_full_bar  = [&](int a) { return bar_base + 8u * (2 * RW_MAX_STAGES + a); };
    auto tmem_empty_bar = [&](int a) { return bar_base + 8u * (2 * RW_MAX_STAGES + 2 + a); };
    const uint32_t b_bar     = bar_base + 8u * (2 * RW_MAX_STAGES + 4);
    const uint32_t tmem_slot = bar_base + 8u * (2 * RW_MAX_STAGES + 5);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA_hi0);
        tma_prefetch_desc(&tmA_lo0);
        tma_prefetch_desc(&tmB_hi);
        tma_prefetch_desc(&tmB_lo);
        for (int s = 0; s < RW_STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tmem_full_bar(a), 1);
            mbar_init(tmem_empty_bar(a), RW_EPI_WARPS);
        }
        mbar_init(b_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 4 * RW_MAX_N); // two accumulator buffers of 2 x (<= 64) columns
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    pdl_wait();
    if (warp == 0) UM_TRACE(5, 0);
    if (p.trace && threadIdx.x == 0) {
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        atomicMin(reinterpret_cast<unsigned long long*>(p.trace) + 5 * 256 + 8, g);
        if (blockIdx.x == 0) p.trace[5 * 256 + 10] = (long long) g;
    }

    const int total_tiles = p.N * p.OH * p.tiles_x;

    if (warp == 0) {
        {
            // weight panel: once per CTA
            if (elect_one()) {
                const int vrows = FKS > 0 ? p.feed_prows : p.kh * p.panels; // (filter row, panel); feed mode: several filter rows per weight row
                mbar_expect_tx(b_bar, (TERMS == 3 ? 2u : 1u) * (uint32_t) vrows * (uint32_t) p.n_blk * 128u);
                for (int v = 0; v < vrows; ++v) {
                    if (TERMS == 3) {
                        tma_load_2d(sB + (2 * v) * p.n_blk * 128, &tmB_hi, b_bar, 0, v * p.ocr);
                        tma_load_2d(sB + (2 * v + 1) * p.n_blk * 128, &tmB_lo, b_bar, 0, v * p.ocr);
                    } else {
                        tma_load_2d(sB + v * p.n_blk * 128, &tmB_hi, b_bar, 0, v * p.ocr); // one plane
                    }
                }
            }
            __syncwarp();
            // activation row segments
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t tx_bytes = (TERMS == 1 ? 1u : 2u) * (p.feed_seg_bytes ? p.feed_seg_bytes : (uint32_t) p.parities * RW_ARR_BYTES);
            if constexpr (FKS > 0) {
                // one contiguous segment per plane and filter row; running pointers, no per-stage address arithmetic
                const uint32_t seg  = p.feed_seg_bytes;
                const size_t pitch  = (size_t) p.feed_w * 4; // fp16 elements per feed row
                const int per_image = p.OH * p.tiles_x;
                int rem = (int) blockIdx.x % per_image, n = (int) blockIdx.x / per_image;
                uint32_t sA = sA0;
                for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                    const int oy = p.tiles_x == 1 ? rem : rem / p.tiles_x, xt = p.tiles_x == 1 ? 0 : rem % p.tiles_x;
                    const size_t off = (((size_t) n * p.feed_h + (oy * 2 - p.pad_y + p.feed_py)) * p.feed_w + 2 * xt * UM_BLOCK_M) * 4;
                    const __half* src_hi = p.feed_hi + off;
                    const __half* src_lo = p.feed_lo + off;
                    for (int ky0 = 0; ky0 < p.kh; ky0 += p.rows_per_stage) {
                        const int rows = min(p.rows_per_stage, p.kh - ky0); // this stage's group of filter rows
                        mbar_wait(empty_bar(stage), phase ^ 1u);
                        if (elect_one()) {
                            if (p.ablate & 2) {
                                mbar_arrive(full_bar(stage));
                            } else {
                                mbar_expect_tx(full_bar(stage), tx_bytes * (uint32_t) rows);
                                const __half* sh = src_hi;
                                const __half* sl = src_lo;
                                uint32_t dst     = sA;
                                for (int r = 0; r < rows; ++r, dst += p.row_bytes, sh += pitch, sl += pitch) {
                                    bulk_load_1d(dst, sh, seg, full_bar(stage));
                                    if (TERMS >= 2) bulk_load_1d(dst + RW_ARR_BYTES, sl, seg, full_bar(stage));
                                }
                            }
                        }
                        __syncwarp();
                        src_hi += pitch * rows, src_lo += pitch * rows;
                        sA += p.stage_bytes;
                        if (++stage == RW_STAGES) stage = 0, phase ^= 1u, sA = sA0;
                    }
                    rem += (int) gridDim.x;
                    while (rem >= per_image) rem -= per_image, ++n;
                }
            } else
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int xt = tile % p.tiles_x, oy = (tile / p.tiles_x) % p.OH, n = tile / (p.tiles_x * p.OH);
                const int ox0 = xt * UM_BLOCK_M;
                for (int ky = 0; ky < p.kh; ++ky) {
                    const int iy = oy * p.stride - p.pad_y + ky; // out of range -> the whole row is zero-filled
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    if (elect_one()) {
                        const uint32_t sA = sA0 + stage * p.stage_bytes;
                        if (p.ablate & 2) {
                            mbar_arrive(full_bar(stage));
                        } else {
                            mbar_expect_tx(full_bar(stage), tx_bytes);
                            tma_load_4d(sA, &tmA_hi0, full_bar(stage), 0, ox0 + p.dmin[0], iy, n);
                            if (TERMS >= 2) tma_load_4d(sA + p.lo_off, &tmA_lo0, full_bar(stage), 0, ox0 + p.dmin[0], iy, n);
                            if (p.parities == 2) {
                                tma_load_4d(sA + RW_ARR_BYTES, &tmA_hi1, full_bar(stage), 0, ox0 + p.dmin[1], iy, n);
                                if (TERMS >= 2) tma_load_4d(sA + p.lo_off + RW_ARR_BYTES, &tmA_lo1, full_bar(stage), 0, ox0 + p.dmin[1], iy, n);
                            }
                        }
                    }
                    __syncwarp();
                    if (++stage == RW_STAGES) stage = 0, phase ^= 1u;
                }
            }
        }
    } else if (warp == 1) {
        mbar_wait(b_bar, 0);
        // see conv_umma_kernel: 3-term = A_hi x [B_hi ; B_lo] + A_lo x B_hi; 2-term = (A_hi + A_lo) x B16; 1-term = A_hi x B_hi
        const uint32_t idesc_cat = TERMS == 3 ? make_idesc(UM_BLOCK_M, 2 * p.n_blk) : make_idesc(UM_BLOCK_M, p.n_blk);
        const uint32_t idesc     = make_idesc(UM_BLOCK_M, p.n_blk);
        if (elect_one()) { // one thread owns the issue loop (see conv_umma_kernel)
            // window descriptor (16-byte address field) offsets of the K steps, relative to the stage's hi plane
            uint32_t koff[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) koff[q] = q < p.ksteps ? (((uint32_t) p.ks_parity[q] * RW_ARR_BYTES + (uint32_t) p.ks_erel[q] * 16u) >> 4) : 0u;
            const uint64_t wdesc0 = make_window_desc(sA0), bdesc0 = make_smem_desc(sB);
            const uint32_t b_panel = (uint32_t) ((TERMS == 3 ? 2 : 1) * p.n_blk * 128) >> 4;  // one [B_hi ; B_lo] (or single-plane) panel (64 K columns)
            const uint32_t b_ky    = b_panel * (uint32_t) p.panels;         // one filter row
            const int last_q      = p.ksteps - 1;
            const uint32_t koff_last = ((uint32_t) p.ks_parity[last_q] * RW_ARR_BYTES + (uint32_t) p.ks_erel[last_q] * 16u) >> 4;
            int stage = 0, it = 0, tr = 0;
            uint32_t phase = 0;
            bool ready     = false;
            const bool no_mma = (p.ablate & 4) != 0;
            const uint64_t lo_off16 = (uint64_t) (p.lo_off >> 4);
            if constexpr (FKS > 0) {
                // FEED mode: K step q of a stage = window start + 2 q pixels pairs (32 B), weights columns 16 q ..; everything a constant offset
                constexpr uint32_t LO16 = RW_ARR_BYTES >> 4;
                constexpr int RPP       = FKS == 1 ? 4 : (FKS == 2 ? 2 : 1); // FeedPlan::rows_per_panel
                const uint32_t stage16  = p.stage_bytes >> 4, row16 = p.row_bytes >> 4;
                const bool tracing      = p.trace != nullptr && blockIdx.x == 0;
                uint64_t a_cur = wdesc0;
                for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                    const int acc = it & 1;
                    mbar_wait(tmem_empty_bar(acc), ((uint32_t) (it >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t) (acc * 2 * RW_MAX_N);
                    uint64_t b_cat = bdesc0;
                    int b_sub      = 0;
                    for (int ky0 = 0; ky0 < p.kh; ky0 += p.rows_per_stage) {
                        const int rows = min(p.rows_per_stage, p.kh - ky0); // the group of filter rows this stage holds
                        if (!ready) mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        if (tracing && tr < 256) p.trace[1 * 256 + tr] = clock64();
                        if (!no_mma) { // first K step of the group, then the look-ahead test, then the rest
                            umma_f16(d_tmem, a_cur, b_cat, idesc_cat, ky0 > 0 ? 1u : 0u);
                            if (TERMS >= 2) umma_f16(d_tmem, a_cur + LO16, b_cat, idesc, 1u);
                        }
                        const int cur        = stage;
                        const bool wrap      = stage == RW_STAGES - 1;
                        uint64_t a_row       = a_cur;
                        phase ^= wrap ? 1u : 0u;
                        stage = wrap ? 0 : stage + 1;
                        a_cur = wrap ? wdesc0 : a_cur + stage16;
                        ready = mbar_test_wait(full_bar(stage), phase); // look-ahead, overlaps with the MMAs already queued
                        for (int r = 0; r < rows; ++r, a_row += row16) {
                            // weights of the next filter row: the next K-column group of the same 128-byte rows, or the next panel
                            const uint64_t b_now = b_cat;
                            if (++b_sub == RPP) b_sub = 0, b_cat += b_panel - (RPP - 1) * (8 / RPP);
                            else b_cat += 8 / RPP;
                            if (no_mma) continue;
#pragma unroll
                            for (int q = 0; q < FKS; ++q) {
                                if (r == 0 && q == 0) continue; // issued above
                                umma_f16(d_tmem, a_row + 2u * q, b_now + 2u * q, idesc_cat, 1u);
                                if (TERMS >= 2) umma_f16(d_tmem, a_row + LO16 + 2u * q, b_now + 2u * q, idesc, 1u);
                            }
                        }
                        umma_commit(empty_bar(cur));
                        if (ky0 + rows == p.kh) umma_commit(tmem_full_bar(acc));
                        if (tracing && tr < 256) p.trace[2 * 256 + tr] = clock64();
                        ++tr;
                    }
                }
            } else
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (uint32_t) (it >> 1) & 1u;
                mbar_wait(tmem_empty_bar(acc), acc_phase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t) (acc * 2 * RW_MAX_N);
                uint64_t b_cat = bdesc0;
                for (int ky = 0; ky < p.kh; ++ky, b_cat += b_ky) {
                    if (!ready) mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    UM_TRACE(1, tr);
                    const uint64_t a0 = wdesc0 + (uint64_t) ((uint32_t) stage * (p.stage_bytes >> 4));
#pragma unroll
                    for (int q = 0; q < 8; ++q) { // K step q lives in weight panel q / 4, columns 16 (q % 4) ..
                        if (q < last_q && !no_mma) {
                            const uint64_t bq = b_cat + (uint64_t) ((q >> 2) * b_panel + 2u * (q & 3));
                            umma_f16(d_tmem, a0 + koff[q], bq, idesc_cat, (ky > 0 || q > 0) ? 1u : 0u);           // -> [hi.hi | hi.lo]
                            if (TERMS >= 2) umma_f16(d_tmem, a0 + lo_off16 + koff[q], bq, idesc, 1u); // lo.hi onto the first block
                        }
                    }
                    const uint64_t b_last = b_cat + (uint64_t) ((last_q >> 2) * b_panel + 2u * (last_q & 3));
                    const int cur = stage;
                    phase ^= (stage == RW_STAGES - 1) ? 1u : 0u;
                    stage = stage == RW_STAGES - 1 ? 0 : stage + 1;
                    ready = mbar_test_wait(full_bar(stage), phase); // look-ahead, overlaps with the MMAs already queued
                    if (!no_mma) {
                        umma_f16(d_tmem, a0 + koff_last, b_last, idesc_cat, (ky > 0 || last_q > 0) ? 1u : 0u);
                        if (TERMS >= 2) umma_f16(d_tmem, a0 + lo_off16 + koff_last, b_last, idesc, 1u);
                    }
                    umma_commit(empty_bar(cur));
                    if (ky == p.kh - 1) umma_commit(tmem_full_bar(acc));
                    UM_TRACE(2, tr);
                    ++tr;
                }
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue: 8 warps, TMEM lane quarter = warp % 4, two interleaved sets of 16-column chunks (see epilogue_tile) ----
        const int q    = warp & 3;
        const int half = (warp - 2) >> 2;
        const int row  = q * 32 + lane;
        EpiArgs e;
        // a 64-channel slab uses the swizzled map, a narrower one the dense map: the host encodes the right one into both slots
        e.o_hi64 = &tmO_hi, e.o_lo64 = &tmO_lo, e.o_hiT = &tmO_hi, e.o_loT = &tmO_lo;
        e.r_hi64 = e.r_lo64 = e.r_hiT = e.r_loT = &tmO_hi;
        e.bias = p.bias, e.n_blk = p.n_blk, e.OC = p.OC, e.act = p.act, e.has_res = 0, e.rows_box = UM_BLOCK_M, e.alpha = p.alpha;
        e.has_lo = TERMS >= 2;
        e.stg = stg, e.res_bar = 0, e.bar_id = 1;
        e.part_src = nullptr, e.part_splits = 0;
        e.no_store = (p.ablate & 8) != 0;
        e.two_stagings = p.stg_bufs == 2;
        uint32_t res_phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (uint32_t) (it >> 1) & 1u;
            const int xt = tile % p.tiles_x, oy = (tile / p.tiles_x) % p.OH, n = tile / (p.tiles_x * p.OH);
            mbar_wait(tmem_full_bar(acc), acc_phase);
            tc_fence_after();
            if (warp == 2) UM_TRACE(3, it);
            e.tmem_empty = tmem_empty_bar(acc);
            e.trace = p.trace, e.trace_seq = it;
            const uint32_t taddr = tmem_base + ((uint32_t) (q * 32) << 16) + (uint32_t) (acc * 2 * RW_MAX_N);
            if (p.ablate & 1) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(e.tmem_empty);
                continue;
            }
            e.stg = stg + (uint32_t) ((it & 1) & (p.stg_bufs - 1)) * UM_STG_BYTES;
            epilogue_tile<RW_EPI_WARPS, TERMS>(e, taddr, 0, xt * UM_BLOCK_M, oy, n, row, half, warp == 2, lane, res_phase);
            if (warp == 2) UM_TRACE(4, it);
        }
        epilogue_drain(warp == 2);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) UM_TRACE(5, 3);
    if (p.trace && threadIdx.x == 0) {
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        atomicMax(reinterpret_cast<unsigned long long*>(p.trace) + 5 * 256 + 9, g);
        if (blockIdx.x == 0) p.trace[5 * 256 + 11] = (long long) g;
    }
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 4 * RW_MAX_N);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Host side: tile-shape selection, tensor maps, launch
// ---------------------------------------------------------------------------------------------------------------
// ---- SNNB_UMMA_TRACE: per-launch timeline of CTA 0 (eager mode only: synchronises around every launch) ----
static bool trace_enabled() {
    static const bool on = getenv("SNNB_UMMA_TRACE") != nullptr;
    return on;
}
static int trace_begin(snnb_context* ctx, long long** out) {
    static long long* d_trace = nullptr;
    if (!d_trace) SNNB_CUDA_OK(cudaMalloc(&d_trace, 6 * 256 * sizeof(long long)));
    SNNB_CUDA_OK(cudaMemsetAsync(d_trace, 0, 6 * 256 * sizeof(long long), ctx->stream));
    const long long big = 0x7fffffffffffffffLL;
    SNNB_CUDA_OK(cudaMemcpyAsync(d_trace + 5 * 256 + 8, &big, sizeof(big), cudaMemcpyHostToDevice, ctx->stream));
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    *out = d_trace;
    return 0;
}
static int trace_end(snnb_context* ctx, const long long* d_trace, const char* header) {
    std::vector<long long> h(6 * 256);
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    SNNB_CUDA_OK(cudaMemcpy(h.data(), d_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    const long long t0 = h[5 * 256];
    fprintf(stderr, "TRACE %s\n", header);
    fprintf(stderr, "  wallclock_ns   all-CTA span %lld | CTA0 entry +%lld exit +%lld\n", h[5 * 256 + 9] - h[5 * 256 + 8], h[5 * 256 + 10] - h[5 * 256 + 8],
            h[5 * 256 + 11] - h[5 * 256 + 8]);
    fprintf(stderr, "  epi_phases (start, +phase1, +wait_read, +barA, +STS, +fence, +barB, +store) per slab:");
    for (int sq = 0; sq < 16 && h[4 * 256 + 64 + 8 * sq]; ++sq) {
        fprintf(stderr, " [");
        for (int k = 1; k < 8; ++k) fprintf(stderr, "%lld ", h[4 * 256 + 64 + 8 * sq + k] ? h[4 * 256 + 64 + 8 * sq + k] - h[4 * 256 + 64 + 8 * sq] : -1);
        fprintf(stderr, "]");
    }
    fprintf(stderr, "\n");
    h[4 * 256 + 64] = 0;
    h[5 * 256 + 4]  = 0; // terminate the clock64 row before the wall-clock slots
    const char* names[6] = {"prod_got_empty", "mma_got_full", "mma_issued", "epi_got_full", "epi_done", "entry_setup_proddone_alldone"};
    for (int r = 0; r < 6; ++r) {
        fprintf(stderr, "  %-14s", names[r]);
        for (int i = 0; i < 256 && (h[r * 256 + i] || (r == 5 && i == 0)); ++i) fprintf(stderr, " %lld", h[r * 256 + i] - t0);
        fprintf(stderr, "\n");
    }
    return 0;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode(snnb_context* ctx) {
    if (!ctx->tmap_encode_fn) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) return nullptr;
        ctx->tmap_encode_fn = fn;
    }
    return reinterpret_cast<EncodeTiledFn>(ctx->tmap_encode_fn);
}

// Tensor maps of an NHWC split-fp16 tensor for the epilogue's TMA stores / residual loads: box = (width channels, tw, th, tn).
static int encode_nhwc_box_maps(EncodeTiledFn encode, const snnb_tensor* t, int width, int tw, int th, int tn, bool swizzle128, CUtensorMap (&maps)[2]) {
    const cuuint64_t dims[4]    = {(cuuint64_t) t->cp, (cuuint64_t) t->w, (cuuint64_t) t->h, (cuuint64_t) t->n};
    const cuuint64_t strides[3] = {(cuuint64_t) t->cp * 2, (cuuint64_t) t->w * t->cp * 2, (cuuint64_t) t->h * t->w * t->cp * 2};
    const cuuint32_t box[4]     = {(cuuint32_t) width, (cuuint32_t) tw, (cuuint32_t) th, (cuuint32_t) tn};
    const cuuint32_t estr[4]    = {1, 1, 1, 1};
    __half* planes[2]    = {t->hi, t->lo ? t->lo : t->hi}; // fp16 storage mode: the lo map is encoded but never used
    for (int i = 0; i < 2; ++i) {
        CUresult r = encode(&maps[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, planes[i], dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        SNNB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(out/residual) failed: %d (cp %d w %d h %d n %d box %d %d %d %d)", (int) r, t->cp, t->w, t->h, t->n,
                     width, tw, th, tn);
    }
    return 0;
}

struct TilePlan {
    int tw = 0, th = 0, tn = 0, tiles_x = 0, tiles_y = 0, tiles_n = 0;
    double eff = 0.0;
};

// Pick the output-pixel box (tw x th x tn <= 128) that wastes the fewest MMA rows. Whole images are stacked (tn > 1)
// only when one image fits in a tile (small feature maps: 7x7, 13x13, 1x1).
static TilePlan plan_tiles(int N, int OH, int OW, int stride) {
    TilePlan best;
    const int max_box = 256 / stride; // TMA boxDim <= 256 (in input elements)
    for (int tw = 1; tw <= std::min(std::min(OW, UM_BLOCK_M), max_box); ++tw) {
        const int max_th = std::min(std::min(OH, UM_BLOCK_M / tw), max_box);
        for (int th = 1; th <= max_th; ++th) {
            int tn = 1;
            if (tw == OW && th == OH) tn = std::min(std::min(N, UM_BLOCK_M / (tw * th)), 256);
            const int tx = (OW + tw - 1) / tw, ty = (OH + th - 1) / th, tnn = (N + tn - 1) / tn;
            const double eff = (double) N * OH * OW / ((double) tx * ty * tnn * UM_BLOCK_M);
            // prefer higher efficiency; on ties prefer wider rows (longer contiguous runs per TMA box row)
            if (eff > best.eff + 1e-9 || (eff > best.eff - 1e-9 && tw > best.tw)) {
                best.tw = tw, best.th = th, best.tn = tn, best.tiles_x = tx, best.tiles_y = ty, best.tiles_n = tnn, best.eff = eff;
            }
        }
    }
    return best;
}

// Output-channel tile width and K split. Measured (profiles/r01_umma_timeline_trace.txt): a K block costs
// max(bytes loaded / ~72 B per clk of L2->SM ingest, MMA issue ~310 clk at n_blk <= 64 / ~420 clk above) and a work item
// another ~7 k clk of ramp-up + last epilogue. A layer takes rounds x that, rounds = ceil(work items / SMs). A narrower
// n_blk re-reads A for more oc tiles but fills more SMs; splitting K (work item = tile x K range, fp32 partials reduced by
// the last arriver, +~9 k clk) fills the GPU when a layer has few tiles and a long K (7x7x512: 128 tiles x 72 K blocks).
// Stream-K split of `tiles` tiles of `num_kb` K blocks over `sms` CTAs: dp whole tiles (full waves), the K blocks of the rest (`units`)
// in `ctas` equal ranges of at least a third of a tile each, so that no tile is cut into more than 4 pieces. False: nothing to cut.
static bool streamk_split(long long tiles, int num_kb, int sms, int& dp, long long& units, int& ctas) {
    dp    = (int) (tiles / sms) * sms;
    units = (tiles - dp) * num_kb;
    const int umin = (num_kb + 2) / 3;
    if (units < umin) return false;
    ctas = (int) std::min<long long>(sms, units / umin);
    return true;
}

struct OcPlan {
    int n_blk = 0, tiles_oc = 0, ksplit = 1, kb_per_split = 0;
    double cost = 1e300; // modelled clocks of the launch
    // stream-K (UmmaParams::sk): whole tiles first, the rest of the tiles' K blocks cut evenly over sk_ctas CTAs
    int sk = 0, sk_dp = 0, sk_ctas = 0;
    long long sk_units = 0;
};
// Tensor-pipe time of one M = 128 tcgen05.mma with N columns (tools/umma_microbench.cu: operand fetch from shared memory, A 4 KB +
// B N x 32 B at 128 B/clk, bounds the narrow shapes): N <= 64: 48 clk, N = 128: 64, N = 256: 128.
static double mma_clk(int n) { return std::max(48.0, n * 0.5); }
static OcPlan plan_oc_ksplit(int OC, int m_tiles, int rows_used, int tile_w, int num_kb, int sm_count, int terms, bool halo = false, bool stream_k = false) {
    OcPlan best;
    double best_cost = 1e300;
    static const int no_split = getenv("SNNB_NO_SPLITK") != nullptr;
    const int max_n = terms == 3 ? UM_MAX_N : UM_MAX_N2;
    const int t_min = (OC + max_n - 1) / max_n, t_max = (OC + 15) / 16;
    for (int t = t_min; t <= t_max; ++t) {
        const int blk = std::min(max_n, round_up((OC + t - 1) / t, 16));
        if (blk * t < OC) continue;
        // boxes narrower than 8 pixels (7x7 maps) move ~20 % fewer bytes per clock through the TMA unit (measured 59 vs 74-77 B/clk)
        const double ingest  = tile_w < 8 ? 58.0 : 72.0;
        // Measured K-block cadences (r02 traces, 3-term): plain 650 clk at n_blk 64 / 811-830 at 128 (the load ring keeps ~3 x 48-64 KB in
        // flight: ~76 B/clk per SM), halo 630 / 890 (tensor-pipe time + ~125 clk: its weight ring runs only a few K blocks ahead). The
        // halo mode therefore wins where the plain mode is ring-bound (n_blk 64) and loses a little where it is MMA-bound (n_blk 128).
        const double a_bytes = (terms == 1 ? 1.0 : 2.0) * rows_used * 128.0, b_bytes = (terms == 3 ? 2.0 : 1.0) * blk * 128;
        const double mma     = terms == 3 ? 4.0 * (mma_clk(2 * blk) + mma_clk(blk)) : 4.0 * terms * mma_clk(blk); // per 64-wide K block
        const double kb_cost = halo ? mma + 125.0 : std::max((a_bytes + b_bytes) / (ingest * 1.05), mma + 45.0);
        for (int sp = 1; sp <= ((no_split || halo) ? 1 : 4); ++sp) {
            if (sp > 1 && (num_kb < 8 * sp)) break; // not worth a reduction for short K
            const int kbps          = (num_kb + sp - 1) / sp;
            if ((sp - 1) * kbps >= num_kb) continue; // an empty split
            const long long items = (long long) m_tiles * t * sp;
            const long long rounds = (items + sm_count - 1) / sm_count;
            const double cost      = (double) rounds * (kbps * kb_cost + 7000.0 + (sp > 1 ? 9000.0 : 0.0));
            if (cost < best_cost * (sp > 1 ? 0.93 : 1.0) - 1e-9) // split only for a clear win
                best_cost = cost, best.cost = cost, best.n_blk = blk, best.tiles_oc = t, best.ksplit = sp, best.kb_per_split = kbps, best.sk = 0;
        }
        // Stream-K: full waves of whole tiles, then the K blocks of the last partial wave's tiles shared evenly by all CTAs (each tile cut
        // into at most 4 pieces, reduced by its last arriver) - instead of a last round that leaves most SMs idle.
        // Opt-in (SNNB_ALGO_TCGEN05_STREAMK / SNNB_SK=1): on ResNet-18's 28x28 and 7x7 layers it measured 3-8 % SLOWER than whole tiles /
        // uniform split-K - the partial dump, the arrival round trip and the last arriver's 3-4 x 64 KB reduction cost more than
        // the idle SMs of the last wave (profiles/README.md).
        static const int env_sk = getenv("SNNB_SK") != nullptr;
        const long long tiles = (long long) m_tiles * t;
        if ((stream_k || env_sk) && !no_split && !halo && num_kb >= 6 && tiles % sm_count != 0) {
            int dp = 0, ctas = 0;
            long long units = 0;
            if (streamk_split(tiles, num_kb, sm_count, dp, units, ctas)) {
                const double u    = std::ceil((double) units / ctas);
                const double cost = (double) (dp / sm_count) * (num_kb * kb_cost + 7000.0) + u * kb_cost + 7000.0 + 4000.0;
                if (cost < best_cost * 0.95 - 1e-9)
                    best_cost = cost, best.cost = cost, best.n_blk = blk, best.tiles_oc = t, best.ksplit = 1, best.kb_per_split = num_kb, best.sk = 1, best.sk_dp = dp,
                    best.sk_ctas = ctas, best.sk_units = units;
            }
        }
        if (blk <= 16) break;
    }
    return best;
}

// fp32 partial tiles + arrival counters of split-K launches. Grow-only, old blocks stay alive until the context dies:
// captured CUDA graphs keep the pointers they were recorded with.
static int ensure_splitk_scratch(snnb_context* ctx, size_t partial_bytes, size_t n_counters) {
    if (partial_bytes > ctx->splitk_bytes) {
        void* pnew = nullptr;
        SNNB_CUDA_OK(cudaMalloc(&pnew, partial_bytes));
        ctx->scratch_blocks.push_back(pnew);
        ctx->splitk_partials = static_cast<float*>(pnew), ctx->splitk_bytes = partial_bytes;
    }
    if (n_counters > ctx->splitk_counter_n) {
        void* pnew = nullptr;
        SNNB_CUDA_OK(cudaMalloc(&pnew, n_counters * sizeof(int)));
        SNNB_CUDA_OK(cudaMemset(pnew, 0, n_counters * sizeof(int)));
        ctx->scratch_blocks.push_back(pnew);
        ctx->splitk_counters = static_cast<int*>(pnew), ctx->splitk_counter_n = n_counters;
    }
    return 0;
}

// How the product is formed (template parameter TERMS of the kernels): the launch's own precision, else the context's default;
// tensors without a lo plane (fp16 storage mode) can only take the 1-term product.
static int conv_terms(const snnb_context* ctx, const ConvArgs& a) {
    if (!a.in->lo || !a.out->lo) return 1;
    const int prec = a.precision >= 0 ? a.precision : ctx->precision;
    return prec == SNNB_PRECISION_FP16W ? 2 : (prec == SNNB_PRECISION_FP16 ? 1 : 3);
}

static bool feed_usable(const ConvArgs& a, FeedPlan& fp);
static bool rowwin_supported(const ConvArgs& a) {
    // small-C stems: IC <= 8 (one 16-byte vector per pixel), stride 1 or 2, <= 8 K steps per filter row, weights packed
    // for exactly this (stride, pad_x), whole panel set resident in smem - in the layout the launch will use (feed mode: one panel)
    RowPlan rp;
    if (!(a.in->cp == 8 && a.w && a.w->w_row_hi && a.w->w_row_lo && a.w->row_stride == a.stride && a.w->row_pad == a.pad_x && a.out->c <= RW_MAX_N &&
          a.residual == nullptr && make_row_plan(a.k, a.stride, a.pad_x, rp) && 128 + rp.span <= RW_BOXW))
        return false;
    FeedPlan fp;
    const int wrows = feed_usable(a, fp) ? (a.k + fp.rows_per_panel - 1) / fp.rows_per_panel : a.k * ((rp.ksteps + 3) / 4); // 128-byte weight rows per channel
    return wrows * 2 * round_up(a.out->c, 16) * 128 <= RW_B_MAX_BYTES;
}

bool conv2d_umma_supported(const ConvArgs& a) {
    if (!a.w || !a.w->w_hi || !a.w->w_lo) return false;
    if (!(a.pad_mode == SNNB_PAD_NONE || a.pad_mode == SNNB_PAD_CONSTANT)) return false; // replicate / reflect: SIMT gather
    if (rowwin_supported(a)) return true;
    if (!(a.stride == 1 || a.stride == 2)) return false; // stride 2 = TMA traversal stride (elementStrides) on W and H
    if (a.in->c < 16) return false; // wider small-C cases the row-GEMM variant cannot take: K would be >75% zero padding
    if (a.k < 1 || a.k > 11) return false;
    if (a.pad_x > 127 || a.pad_y > 127) return false;
    return true;
}

// halo mode (3x3, stride 1): 8 x 16-pixel tiles whose nine taps share one halo load; taken when the cost model prefers it to the plain
// plan of cost `plain_cost` (fewer bytes per K block against the MMA rows lost where 8 / 16 do not divide the feature map)
static bool halo_plan(const snnb_context* ctx, const ConvArgs& a, int cblocks, int terms, double plain_cost, OcPlan& hp) {
    static const bool no_halo = getenv("SNNB_NO_HALO") != nullptr;
    if (no_halo || a.k != 3 || a.stride != 1 || a.pad_x > 1 || a.pad_y > 1) return false;
    const int hx = (a.out->w + HL_TW - 1) / HL_TW, hy = (a.out->h + HL_TH - 1) / HL_TH;
    hp = plan_oc_ksplit(a.out->c, hx * hy * a.out->n, UM_BLOCK_M, HL_TW, 9 * cblocks, ctx->sm_count, terms, true);
    return hp.n_blk > 0 && hp.cost < plain_cost;
}

bool conv2d_umma_fold_supported(const snnb_context* ctx, const ConvArgs& a) {
    if (!a.shortcut || a.residual || !conv2d_umma_supported(a) || rowwin_supported(a)) return false;
    // stride <= 2 keeps the shortcut's box (tw * s, th * s with tw, th <= 128) within TMA's 256 elements per dimension
    if (!(a.sc_stride == 1 || a.sc_stride == 2) || a.shortcut->n != a.out->n || !a.shortcut->lo != !a.in->lo) return false;
    const TilePlan tp = plan_tiles(a.out->n, a.out->h, a.out->w, a.stride);
    if (tp.tw <= 0) return false;
    // the layer as it would run unfolded: a layer the halo mode serves better keeps its own launch (the fold is plain mode only)
    const int cblocks = (a.in->c + UM_BLOCK_K - 1) / UM_BLOCK_K, terms = conv_terms(ctx, a);
    const OcPlan op   = plan_oc_ksplit(a.out->c, tp.tiles_x * tp.tiles_y * tp.tiles_n, tp.tw * tp.th * tp.tn, tp.tw, a.k * a.k * cblocks, ctx->sm_count, terms, false,
                                       a.stream_k);
    OcPlan hp;
    return op.n_blk > 0 && !halo_plan(ctx, a, cblocks, terms, op.cost, hp);
}

enum { ATTR_UMMA = 1u, ATTR_ROWWIN = 2u, ATTR_DW1 = 4u, ATTR_DW2 = 8u }; // bits of snnb_context::func_attr_mask

typedef void (*RowWinKernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap,
                             const CUtensorMap, const RowWinParams);
template <int TERMS> static RowWinKernel rowwin_kernel_fks(int fks) {
    switch (fks) {
    case 1: return conv_rowwin_kernel<TERMS, 1>;
    case 2: return conv_rowwin_kernel<TERMS, 2>;
    case 3: return conv_rowwin_kernel<TERMS, 3>;
    case 4: return conv_rowwin_kernel<TERMS, 4>;
    default: return conv_rowwin_kernel<TERMS, 0>;
    }
}
static RowWinKernel rowwin_kernel_of(int terms, int fks) { return terms == 3 ? rowwin_kernel_fks<3>(fks) : (terms == 2 ? rowwin_kernel_fks<2>(fks) : rowwin_kernel_fks<1>(fks)); }

// FEED mode: the input tensor carries the compact 4-channel copy this layer's weights were packed for, and it is large enough
static bool feed_usable(const ConvArgs& a, FeedPlan& fp) {
    const snnb_tensor* in = a.in;
    if (!in->feed_hi || !a.w->w_feed_hi || !a.w->w_feed_lo || a.w->feed_pad != a.pad_x) return false;
    if (!make_feed_plan(a.k, a.stride, a.pad_x, in->c, fp) || fp.px != in->feed_px || in->feed_py != a.pad_y) return false;
    const int tiles_x = (a.out->w + UM_BLOCK_M - 1) / UM_BLOCK_M;
    return in->feed_w >= 2 * (tiles_x * UM_BLOCK_M - 1) + 2 * fp.nch && in->feed_h >= 2 * (a.out->h - 1) + a.k &&
           (254 + 2 * fp.nch) * 8 <= RW_ARR_BYTES;
}

static int launch_conv2d_rowwin(snnb_context* ctx, const ConvArgs& a, EncodeTiledFn encode) {
    const snnb_tensor* in = a.in;
    snnb_tensor* out      = a.out;
    RowPlan rp;
    SNNB_REQUIRE(make_row_plan(a.k, a.stride, a.pad_x, rp), "launch_conv2d_rowwin: no row plan");
    FeedPlan fp;
    const bool feed = feed_usable(a, fp);
    SNNB_REQUIRE(feed || !in->feed_only, "launch_conv2d_rowwin: the input tensor only exists as a stem feed, which this launch cannot read");
    if (feed) { // one dense segment per plane, K steps at consecutive 32-byte offsets
        rp.parities = 1, rp.ksteps = fp.ksteps;
        for (int q = 0; q < fp.ksteps; ++q) rp.ks_parity[q] = 0, rp.ks_erel[q] = 2 * q;
    }
    ctx->last_kernel = feed ? "conv_rowwin_kernel<feed>" : "conv_rowwin_kernel";
    RowWinParams p;
    p.out_hi = out->hi, p.out_lo = out->lo, p.bias = a.w->bias;
    p.N = out->n, p.OH = out->h, p.OW = out->w, p.OC = out->c, p.OCp = out->cp;
    p.n_blk = round_up(out->c, 16), p.ocr = a.w->ocr;
    p.kh = a.k, p.stride = a.stride, p.pad_y = a.pad_y;
    p.tiles_x  = (out->w + UM_BLOCK_M - 1) / UM_BLOCK_M;
    p.parities = rp.parities, p.dmin[0] = rp.dmin[0], p.dmin[1] = rp.dmin[1];
    p.ksteps   = rp.ksteps, p.panels = (rp.ksteps + 3) / 4;
    for (int q = 0; q < 8; ++q) p.ks_parity[q] = q < rp.ksteps ? rp.ks_parity[q] : 0, p.ks_erel[q] = q < rp.ksteps ? rp.ks_erel[q] : 0;
    p.act = a.act, p.alpha = a.alpha;
    static const int rw_ablate = getenv("SNNB_UMMA_ABLATE") ? atoi(getenv("SNNB_UMMA_ABLATE")) : 0;
    p.ablate                   = rw_ablate;
    p.feed_hi = in->feed_hi, p.feed_lo = in->feed_lo, p.feed_h = in->feed_h, p.feed_w = in->feed_w, p.feed_py = in->feed_py;
    p.feed_seg_bytes = feed ? (uint32_t) (254 + 2 * fp.nch) * 8u : 0u;
    const int terms = conv_terms(ctx, a);
    p.lo_off      = (uint32_t) p.parities * RW_ARR_BYTES;
    p.row_bytes   = (terms == 1 ? 1u : 2u) * p.lo_off;
    // feed mode: ceil(kh / 4) groups of filter rows, as even as possible (7 -> 4 + 3, 3 -> 3, 9 -> 3 + 3 + 3)
    static const int one_row = getenv("SNNB_FEED_ONE_ROW") != nullptr;
    p.rows_per_stage = (feed && !one_row) ? (a.k + (a.k + 3) / 4 - 1) / ((a.k + 3) / 4) : 1;
    p.stage_bytes    = (uint32_t) p.rows_per_stage * p.row_bytes;
    p.feed_prows  = feed ? (a.k + fp.rows_per_panel - 1) / fp.rows_per_panel : 0;
    p.b_bytes     = (uint32_t) round_up((terms == 3 ? 2 : 1) * (feed ? p.feed_prows : a.k * p.panels) * p.n_blk * 128, 1024);
    // a second staging buffer when the ring keeps >= 2 stages beside it (one slab per tile: n_blk <= 64 always holds here)
    static const int one_stg = getenv("SNNB_ROWWIN_ONE_STAGING") != nullptr;
    const int ring_room      = RW_SMEM_BYTES - 1024 - RW_BAR_BYTES - (int) p.b_bytes;
    p.stg_bufs    = (!one_stg && (ring_room - 2 * UM_STG_BYTES) / (int) p.stage_bytes >= 2) ? 2 : 1;
    p.stages      = std::min(RW_MAX_STAGES, (ring_room - p.stg_bufs * UM_STG_BYTES) / (int) p.stage_bytes);
    SNNB_REQUIRE(p.stages >= 2, "launch_conv2d_rowwin: weight panels of %u bytes leave no room for the activation ring", p.b_bytes);

    // A: per plane and column parity a 4-D view (8 ch | de-interleaved pixel index | row | image) of the NHWC plane
    CUtensorMap tmA[4], tmB[2];
    for (int plane = 0; plane < 2; ++plane)
        for (int par = 0; par < 2; ++par) {
            const int pp = par < rp.parities ? par : 0; // unused maps alias parity 0 (kernel never issues them)
            __half* base = ((plane && in->lo) ? in->lo : in->hi) + (size_t) pp * 8; // half-precision storage mode: the lo maps are never issued
            const int wp        = (in->w - pp + a.stride - 1) / a.stride; // pixels of this parity per row
            const cuuint64_t dims[4]    = {8, (cuuint64_t) (wp > 0 ? wp : 1), (cuuint64_t) in->h, (cuuint64_t) in->n};
            const cuuint64_t strides[3] = {(cuuint64_t) a.stride * 16, (cuuint64_t) in->w * 16, (cuuint64_t) in->h * in->w * 16};
            const cuuint32_t box[4]     = {8, (cuuint32_t) RW_BOXW, 1, 1};
            const cuuint32_t estr[4]    = {1, 1, 1, 1};
            CUresult r = encode(&tmA[plane * 2 + par], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            SNNB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(A, rowwin) failed: %d", (int) r);
        }
    {
        const cuuint64_t dims[2]    = {64, (cuuint64_t) (feed ? (a.k + fp.rows_per_panel - 1) / fp.rows_per_panel : a.k * p.panels) * a.w->ocr}; // [ky][panel][OCr] rows of 64 K columns
        const cuuint64_t strides[1] = {128};
        const cuuint32_t box[2]     = {64, (cuuint32_t) p.n_blk};
        const cuuint32_t estr[2]    = {1, 1};
        void* planes[2] = {(void*) (feed ? a.w->w_feed_hi : a.w->w_row_hi), (void*) (feed ? a.w->w_feed_lo : a.w->w_row_lo)}; // 2-term: the hi plane alone = fp16_rn(w)
        for (int i = 0; i < 2; ++i) {
            CUresult r = encode(&tmB[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, planes[i], dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            SNNB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(B, rowwin) failed: %d", (int) r);
        }
    }
    CUtensorMap tmO[2];
    if (encode_nhwc_box_maps(encode, out, p.n_blk, UM_BLOCK_M, 1, 1, p.n_blk == 64, tmO)) return 2;
    if (!(ctx->func_attr_mask & ATTR_ROWWIN)) {
        for (int t = 1; t <= 3; ++t)
            for (int f = 0; f <= 4; ++f) SNNB_CUDA_OK(cudaFuncSetAttribute(rowwin_kernel_of(t, f), cudaFuncAttributeMaxDynamicSharedMemorySize, RW_SMEM_BYTES));
        ctx->func_attr_mask |= ATTR_ROWWIN;
    }
    const int total_tiles = p.N * p.OH * p.tiles_x;
    const int grid        = std::min(total_tiles, ctx->sm_count);
    p.trace = nullptr;
    if (trace_enabled() && trace_begin(ctx, &p.trace)) return 1;
    auto* kern = rowwin_kernel_of(terms, feed ? fp.ksteps : 0);
    const cudaError_t le = launch_k_pdl(kern, dim3(grid), dim3(RW_THREADS), RW_SMEM_BYTES, ctx->stream, tmA[0], tmA[1], tmA[2], tmA[3], tmB[0], tmB[1], tmO[0], tmO[1], p);
    if (p.trace) {
        char hdr[256];
        snprintf(hdr, sizeof hdr, "rowwin%s k%d s%d IC%d OC%d out %dx%dx%d n_blk %d tiles %d grid %d kh %d ksteps %d terms %d", feed ? "<feed>" : "", a.k, a.stride, a.in->c,
                 a.out->c, a.out->n, a.out->h, a.out->w, p.n_blk, total_tiles, grid, p.kh, p.ksteps, terms);
        if (trace_end(ctx, p.trace, hdr)) return 1;
    }
    cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("conv_rowwin_kernel launch failed: %s", cudaGetErrorString(e));
        return 1;
    }
    ctx->launches++;
    return 0;
}

int launch_conv2d_umma(snnb_context* ctx, const ConvArgs& a) {
    EncodeTiledFn encode = get_encode(ctx);
    SNNB_REQUIRE(encode, "launch_conv2d_umma: cuTensorMapEncodeTiled is unavailable in this driver");
    if (rowwin_supported(a)) {
        SNNB_REQUIRE(!a.shortcut, "launch_conv2d_umma: a folded shortcut needs the plain tensor-core kernel, not the row-window kernel");
        return launch_conv2d_rowwin(ctx, a, encode);
    }
    SNNB_REQUIRE(!a.in->feed_only && !(a.shortcut && a.shortcut->feed_only), "launch_conv2d_umma: the input tensor only exists as a stem feed, which this launch cannot read");
    SNNB_REQUIRE(!(a.shortcut && a.residual), "launch_conv2d_umma: a folded shortcut and a residual operand are exclusive");
    SNNB_REQUIRE(!a.shortcut || ((a.sc_stride == 1 || a.sc_stride == 2) && a.shortcut->n == a.out->n), "launch_conv2d_umma: unsupported shortcut (stride %d)",
                 a.sc_stride);
    const snnb_tensor* in = a.in;
    snnb_tensor* out      = a.out;
    UmmaParams p;
    p.out_hi = out->hi, p.out_lo = out->lo;
    p.res_hi = a.residual ? a.residual->hi : nullptr, p.res_lo = a.residual ? a.residual->lo : nullptr;
    p.has_res = a.residual != nullptr;
    p.bias    = a.w->bias;
    p.N = out->n, p.OH = out->h, p.OW = out->w, p.OC = out->c, p.OCp = out->cp;
    const TilePlan tp = plan_tiles(out->n, out->h, out->w, a.stride);
    SNNB_REQUIRE(tp.tw > 0, "launch_conv2d_umma: no tile plan");
    p.tw = tp.tw, p.th = tp.th, p.tn = tp.tn, p.rows_used = tp.tw * tp.th * tp.tn;
    p.tiles_x = tp.tiles_x, p.tiles_y = tp.tiles_y, p.tiles_n = tp.tiles_n;
    p.ksize = a.k, p.stride = a.stride, p.pad_x = a.pad_x, p.pad_y = a.pad_y;
    p.cblocks = (in->c + UM_BLOCK_K - 1) / UM_BLOCK_K;
    p.sc_cblocks = a.shortcut ? (a.shortcut->c + UM_BLOCK_K - 1) / UM_BLOCK_K : 0, p.sc_stride = a.shortcut ? a.sc_stride : 1;
    const int num_kb = a.k * a.k * p.cblocks + p.sc_cblocks;
    const int terms = conv_terms(ctx, a);
    p.has_lo        = out->lo != nullptr;
    p.b_stages = 0, p.b_stage_bytes = 0;
    OcPlan op       = plan_oc_ksplit(out->c, tp.tiles_x * tp.tiles_y * tp.tiles_n, p.rows_used, tp.tw, num_kb, ctx->sm_count, terms, false, a.stream_k);
    OcPlan hp;
    const bool halo = !a.shortcut && halo_plan(ctx, a, p.cblocks, terms, op.cost, hp); // the halo producer has no shortcut operand
    if (halo) {
        op              = hp;
        p.b_stage_bytes = (terms == 3 ? 2 : 1) * op.n_blk * 128 <= UM_B_BYTES ? UM_B_BYTES : 2 * UM_B_BYTES; // 16 KB when a stage fits, else 32 KB
        p.b_stages      = HL_B_RING_BYTES / p.b_stage_bytes;
        p.tw = HL_TW, p.th = HL_TH, p.tn = 1, p.rows_used = UM_BLOCK_M;
        p.tiles_x = (out->w + HL_TW - 1) / HL_TW, p.tiles_y = (out->h + HL_TH - 1) / HL_TH, p.tiles_n = out->n;
    }
    SNNB_REQUIRE(op.n_blk > 0, "launch_conv2d_umma: no output-channel plan");
    p.n_blk = op.n_blk, p.tiles_oc = op.tiles_oc, p.ksplit = op.ksplit, p.kb_per_split = op.kb_per_split;
    p.sk = halo ? 0 : op.sk, p.sk_dp = op.sk_dp, p.sk_ctas = op.sk_ctas, p.sk_units = op.sk_units;
    p.partials = nullptr, p.counters = nullptr;
    if (!ctx->sched_counter) { // created by the first (eager) launch; graph capture replays use the same word
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        SNNB_CUDA_OK(cudaStreamIsCapturing(ctx->stream, &cap));
        SNNB_REQUIRE(cap == cudaStreamCaptureStatusNone, "launch_conv2d_umma: the scheduler counter must be allocated by an eager pass before graph capture");
        void* pnew = nullptr;
        SNNB_CUDA_OK(cudaMalloc(&pnew, 256));
        SNNB_CUDA_OK(cudaMemset(pnew, 0, 256));
        ctx->scratch_blocks.push_back(pnew);
        ctx->sched_counter = static_cast<int*>(pnew);
    }
    p.sched_counter = ctx->sched_counter;
    if (p.ksplit > 1 || p.sk) {
        // partial-tile slots: split-K [tile][split]; stream-K [tile past sk_dp][4 pieces]
        const size_t tiles = p.sk ? (size_t) p.tiles_x * p.tiles_y * p.tiles_n * p.tiles_oc - p.sk_dp : (size_t) p.tiles_x * p.tiles_y * p.tiles_n * p.tiles_oc;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        SNNB_CUDA_OK(cudaStreamIsCapturing(ctx->stream, &cap));
        const size_t need = tiles * (p.sk ? 4 : p.ksplit) * UM_BLOCK_M * p.n_blk * sizeof(float);
        SNNB_REQUIRE(cap == cudaStreamCaptureStatusNone || (need <= ctx->splitk_bytes && tiles <= ctx->splitk_counter_n),
                     "launch_conv2d_umma: split-K scratch must be allocated by an eager pass before graph capture");
        if (ensure_splitk_scratch(ctx, need, tiles)) return 1;
        p.partials = ctx->splitk_partials, p.counters = ctx->splitk_counters;
    }
    p.ICp     = round_up(in->c, 8);
    p.act = a.act, p.alpha = a.alpha;
    static const int ablate = getenv("SNNB_UMMA_ABLATE") ? atoi(getenv("SNNB_UMMA_ABLATE")) : 0;
    p.ablate                = ablate;
    const int kp_want = a.k * a.k * p.ICp + (a.shortcut ? round_up(a.shortcut->c, 8) : 0); // [taps | shortcut] columns
    SNNB_REQUIRE(a.w->kp == kp_want, "launch_conv2d_umma: packed weights do not match (kp %d vs %d)", a.w->kp, kp_want);

    // A operand maps: box = the output tile's pixels at traversal stride s (halo mode: the halo tile); channel tail zero-filled
    auto encode_a = [&](const snnb_tensor* t, int s, int bw, int bh, CUtensorMap (&maps)[2]) {
        const cuuint64_t dims[4]    = {(cuuint64_t) t->c, (cuuint64_t) t->w, (cuuint64_t) t->h, (cuuint64_t) t->n};
        const cuuint64_t strides[3] = {(cuuint64_t) t->cp * 2, (cuuint64_t) t->w * t->cp * 2, (cuuint64_t) t->h * t->w * t->cp * 2};
        const cuuint32_t box[4]     = {(cuuint32_t) UM_BLOCK_K, (cuuint32_t) bw, (cuuint32_t) bh, (cuuint32_t) p.tn};
        const cuuint32_t estr[4]    = {1, (cuuint32_t) s, (cuuint32_t) s, 1};
        __half* planes[2]    = {t->hi, t->lo ? t->lo : t->hi}; // fp16 storage mode: the lo map is never issued
        for (int i = 0; i < 2; ++i) {
            CUresult r = encode(&maps[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, planes[i], dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            SNNB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(A) failed: %d (dims %d %d %d %d box %u %u %u %u)", (int) r, t->c, t->w, t->h, t->n, box[0],
                         box[1], box[2], box[3]);
        }
        return 0;
    };
    CUtensorMap tmA[2], tmB[2], tmS[2];
    if (encode_a(in, a.stride, halo ? HL_W : p.tw * a.stride, halo ? HL_H : p.th * a.stride, tmA)) return 2;
    if (!a.shortcut) {
        tmS[0] = tmA[0], tmS[1] = tmA[1]; // never issued
    } else if (encode_a(a.shortcut, a.sc_stride, p.tw * a.sc_stride, p.th * a.sc_stride, tmS)) {
        return 2;
    }
    {
        const cuuint64_t dims[2]    = {(cuuint64_t) a.w->kp, (cuuint64_t) a.w->ocr};
        const cuuint64_t strides[1] = {(cuuint64_t) a.w->kp * 2};
        const cuuint32_t box[2]     = {(cuuint32_t) UM_BLOCK_K, (cuuint32_t) p.n_blk};
        const cuuint32_t estr[2]    = {1, 1};
        void* planes[2]             = {(void*) a.w->w_hi, (void*) a.w->w_lo}; // the 2-term product uses the hi plane alone: fp16_rn(w)
        for (int i = 0; i < 2; ++i) {
            CUresult r = encode(&tmB[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, planes[i], dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            SNNB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(B) failed: %d (kp %d ocr %d n_blk %d)", (int) r, a.w->kp, a.w->ocr, p.n_blk);
        }
    }
    // epilogue maps: full 64-channel slabs (swizzled) and the tail slab (n_blk % 64 channels, dense)
    CUtensorMap tmO64[2], tmOT[2], tmR64[2], tmRT[2];
    {
        const int wT = p.n_blk % 64;
        const snnb_tensor* res = a.residual ? a.residual : out;
        if (encode_nhwc_box_maps(encode, out, p.n_blk >= 64 ? 64 : wT, p.tw, p.th, p.tn, p.n_blk >= 64, tmO64)) return 2;
        if (encode_nhwc_box_maps(encode, out, wT ? wT : 64, p.tw, p.th, p.tn, wT == 0, tmOT)) return 2;
        if (encode_nhwc_box_maps(encode, res, p.n_blk >= 64 ? 64 : wT, p.tw, p.th, p.tn, p.n_blk >= 64, tmR64)) return 2;
        if (encode_nhwc_box_maps(encode, res, wT ? wT : 64, p.tw, p.th, p.tn, wT == 0, tmRT)) return 2;
    }
    if (!(ctx->func_attr_mask & ATTR_UMMA)) {
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES, false, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES, false, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES, false, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES - 1, true, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES_SPLIT));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES - 1, true, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES_SPLIT));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES - 1, true, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES_SPLIT));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<HL_B_STAGES, false, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, HL_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<HL_B_STAGES, false, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, HL_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<HL_B_STAGES, false, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, HL_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES, false, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES, false, 2, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES));
        SNNB_CUDA_OK(cudaFuncSetAttribute(conv_umma_kernel<UM_STAGES, false, 3, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_SMEM_BYTES));
        ctx->func_attr_mask |= ATTR_UMMA;
    }
    const int total_tiles = p.tiles_x * p.tiles_y * p.tiles_n * p.tiles_oc;
    const int grid        = p.sk ? (p.sk_dp > 0 ? ctx->sm_count : p.sk_ctas) : std::min(total_tiles * p.ksplit, ctx->sm_count);
    // short K loop (1x1 convolutions): the layer runs at the speed of the epilogue -> two independent epilogue groups
    static const bool no_split_epi = getenv("SNNB_NO_SPLIT_EPI") != nullptr;
    const bool split_epi           = !halo && !no_split_epi && !p.sk && p.ksplit == 1 && num_kb <= 3 && total_tiles >= 2 * grid;
    ctx->last_kernel = halo ? "conv_umma_kernel<halo>"
                            : (split_epi ? "conv_umma_kernel<short-K>" : (p.sk ? "conv_umma_kernel<stream-K>" : (p.ksplit > 1 ? "conv_umma_kernel<split-K>" : "conv_umma_kernel")));
    p.trace = nullptr;
    if (trace_enabled() && trace_begin(ctx, &p.trace)) return 1;
    auto* k_split = terms == 3 ? conv_umma_kernel<UM_STAGES - 1, true, 3, false> : (terms == 2 ? conv_umma_kernel<UM_STAGES - 1, true, 2, false> : conv_umma_kernel<UM_STAGES - 1, true, 1, false>);
    auto* k_plain = p.sk ? (terms == 3 ? conv_umma_kernel<UM_STAGES, false, 3, false, true>
                                       : (terms == 2 ? conv_umma_kernel<UM_STAGES, false, 2, false, true> : conv_umma_kernel<UM_STAGES, false, 1, false, true>) )
                         : (terms == 3 ? conv_umma_kernel<UM_STAGES, false, 3, false> : (terms == 2 ? conv_umma_kernel<UM_STAGES, false, 2, false> : conv_umma_kernel<UM_STAGES, false, 1, false>) );
    auto* k_halo  = terms == 3 ? conv_umma_kernel<HL_B_STAGES, false, 3, true> : (terms == 2 ? conv_umma_kernel<HL_B_STAGES, false, 2, true> : conv_umma_kernel<HL_B_STAGES, false, 1, true>);
    const cudaError_t le =
        halo      ? launch_k_pdl(k_halo, dim3(grid), dim3(UM_THREADS), HL_SMEM_BYTES, ctx->stream, tmA[0], tmA[1], tmB[0], tmB[1], tmO64[0], tmO64[1], tmOT[0], tmOT[1], tmR64[0],
                                 tmR64[1], tmRT[0], tmRT[1], tmS[0], tmS[1], p)
        : split_epi ? launch_k_pdl(k_split, dim3(grid), dim3(UM_THREADS), UM_SMEM_BYTES_SPLIT, ctx->stream, tmA[0], tmA[1], tmB[0], tmB[1], tmO64[0], tmO64[1], tmOT[0], tmOT[1],
                                 tmR64[0], tmR64[1], tmRT[0], tmRT[1], tmS[0], tmS[1], p)
                  : launch_k_pdl(k_plain, dim3(grid), dim3(UM_THREADS), UM_SMEM_BYTES, ctx->stream, tmA[0], tmA[1], tmB[0], tmB[1], tmO64[0], tmO64[1], tmOT[0], tmOT[1], tmR64[0],
                                 tmR64[1], tmRT[0], tmRT[1], tmS[0], tmS[1], p);
    if (p.trace) {
        char hdr[256];
        snprintf(hdr, sizeof hdr, "conv k%d s%d IC%d OC%d out %dx%dx%d n_blk %d tiles %d grid %d num_kb %d ksplit %d terms %d halo %d", a.k, a.stride, in->c, out->c, out->n,
                 out->h, out->w, p.n_blk, total_tiles, grid, num_kb, split_epi ? -1 : (p.sk ? -2 : p.ksplit), terms, (int) halo); // ksplit -1 = split-epilogue variant, -2 = stream-K
        if (trace_end(ctx, p.trace, hdr)) return 1;
    }
    cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("conv_umma_kernel launch failed: %s", cudaGetErrorString(e));
        return 1;
    }
    ctx->launches++;
    return 0;
}


// ---------------------------------------------------------------------------------------------------------------
// Depthwise 3x3 (stride 1 / 2), TMA-staged + register-tiled (shadertemplate_vk_depthwise.comp:64-139).
//
// HBM-bound work: every input byte should cross the memory system once. A persistent CTA walks tiles of
// TH x TW output pixels x 64 channels; for each tile ONE TMA box load per plane brings the (TH-1)*S+3 x (TW-1)*S+3
// input patch (128-byte pixel rows, no swizzle; out-of-image pixels and channels >= C are zero-filled = the zero padding)
// into a 3-deep shared-memory ring, so loads of the next tiles are in flight while this one is computed. A thread owns
// 8 channels (one 16-byte piece of the pixel row) and TXT consecutive output columns and streams the patch rows through
// registers (stride 1: 18 pixel loads for 4 outputs). A warp reads 4 pixel rows x 128 B per instruction: conflict-free.
// Outputs go straight to global memory: a warp writes 4 full 128-byte lines per plane.
// ---------------------------------------------------------------------------------------------------------------
constexpr int DW_THREADS = 256;
constexpr int DW_STAGES  = 2;
template <int S> struct DwTile {
    static constexpr int TW = S == 1 ? 16 : 8, TH = S == 1 ? 8 : 4; // output pixels per tile: 128 / 32
    static constexpr int TXT = S == 1 ? 4 : 1;                      // output columns per thread
    static constexpr int IW = (TW - 1) * S + 3, IH = (TH - 1) * S + 3;
    static constexpr int PLANE_BYTES = IW * IH * 128;
    static constexpr int STAGE_BYTES = 2 * PLANE_BYTES;
    static constexpr int SMEM_BYTES  = DW_STAGES * STAGE_BYTES + 128 /*alignment*/ + 64 /*barriers*/;
};
struct DwTmaParams {
    __half* out_hi;
    __half* out_lo;
    const float* w;    // [9][Cp]
    const float* bias; // [Cp + padding]
    int N, OH, OW, C, Cp;
    int pad_x, pad_y;
    int tiles_x, tiles_y, chunks;
    int act;
    float alpha;
};

template <int S>
__global__ void __launch_bounds__(DW_THREADS, 2) depthwise_tma_kernel(const __grid_constant__ CUtensorMap tmI_hi, const __grid_constant__ CUtensorMap tmI_lo, const DwTmaParams p) {
    using T = DwTile<S>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 127u) & ~127u;
    const uint32_t bar_base  = smem_base + DW_STAGES * T::STAGE_BYTES;
    const int tid = threadIdx.x, warp = tid >> 5;
    pdl_trigger();
    if (tid == 0) {
        tma_prefetch_desc(&tmI_hi);
        tma_prefetch_desc(&tmI_lo);
        for (int s = 0; s < DW_STAGES; ++s) mbar_init(bar_base + 8u * s, 1);
        fence_barrier_init();
    }
    __syncthreads();
    pdl_wait();

    const int sp_tiles = p.N * p.tiles_y * p.tiles_x;
    const int total    = sp_tiles * p.chunks; // chunk is the slowest index: a CTA's consecutive tiles share its weights
    auto issue = [&](int tile, int stage) {   // one thread
        const int chunk = tile / sp_tiles, sp = tile - chunk * sp_tiles;
        const int tx = sp % p.tiles_x, ty = (sp / p.tiles_x) % p.tiles_y, n = sp / (p.tiles_x * p.tiles_y);
        const uint32_t dst = smem_base + stage * T::STAGE_BYTES, bar = bar_base + 8u * stage;
        mbar_expect_tx(bar, T::STAGE_BYTES);
        tma_load_4d(dst, &tmI_hi, bar, chunk * 64, tx * T::TW * S - p.pad_x, ty * T::TH * S - p.pad_y, n);
        tma_load_4d(dst + T::PLANE_BYTES, &tmI_lo, bar, chunk * 64, tx * T::TW * S - p.pad_x, ty * T::TH * S - p.pad_y, n);
    };
    if (tid == 0)
        for (int j = 0; j < DW_STAGES; ++j) {
            const int tile = blockIdx.x + j * gridDim.x;
            if (tile < total) issue(tile, j);
        }

    const int cg  = tid & 7, pt = tid >> 3;                                            // 16-byte channel piece, pixel-thread 0..31
    const int tyl = S == 1 ? (pt >> 2) : (pt >> 3), txl = S == 1 ? (pt & 3) * 4 : (pt & 7); // first output (row, col) in the tile
    const float slope   = (p.act == SNNB_ACT_RELU || p.act == SNNB_ACT_RELU6) ? 0.0f : (p.act == SNNB_ACT_LEAKY_RELU ? p.alpha : 1.0f);
    const float hi_clip = p.act == SNNB_ACT_RELU6 ? 6.0f : __int_as_float(0x7f800000);
    const bool fast_act = p.act == SNNB_ACT_NONE || p.act == SNNB_ACT_RELU || p.act == SNNB_ACT_RELU6 || p.act == SNNB_ACT_LEAKY_RELU;

    float wreg[9][8], breg[8];
    int cur_chunk = -1;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
        const int stage = it % DW_STAGES;
        const int chunk = tile / sp_tiles, sp = tile - chunk * sp_tiles;
        const int tx = sp % p.tiles_x, ty = (sp / p.tiles_x) % p.tiles_y, n = sp / (p.tiles_x * p.tiles_y);
        const int c = chunk * 64 + cg * 8;
        if (chunk != cur_chunk) { // this thread's 8 channels of the folded weights and bias
            cur_chunk = chunk;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;
                if (c < p.Cp) {
                    w0 = __ldg(reinterpret_cast<const float4*>(p.w + (size_t) t * p.Cp + c));
                    w1 = __ldg(reinterpret_cast<const float4*>(p.w + (size_t) t * p.Cp + c) + 1);
                }
                wreg[t][0] = w0.x, wreg[t][1] = w0.y, wreg[t][2] = w0.z, wreg[t][3] = w0.w;
                wreg[t][4] = w1.x, wreg[t][5] = w1.y, wreg[t][6] = w1.z, wreg[t][7] = w1.w;
            }
            float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
            if (c < p.Cp) {
                b0 = __ldg(reinterpret_cast<const float4*>(p.bias + c));
                b1 = __ldg(reinterpret_cast<const float4*>(p.bias + c) + 1);
            }
            breg[0] = b0.x, breg[1] = b0.y, breg[2] = b0.z, breg[3] = b0.w, breg[4] = b1.x, breg[5] = b1.y, breg[6] = b1.z, breg[7] = b1.w;
        }
        mbar_wait(bar_base + 8u * stage, (uint32_t) (it / DW_STAGES) & 1u);
        const uint32_t src = smem_base + stage * T::STAGE_BYTES + (uint32_t) cg * 16u;

        float acc[T::TXT][8];
#pragma unroll
        for (int t = 0; t < T::TXT; ++t)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[t][j] = breg[j];
        constexpr int COLS = S * (T::TXT - 1) + 3;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
            for (int cx = 0; cx < COLS; ++cx) {
                const uint32_t a = src + (uint32_t) (((tyl * S + ky) * T::IW + txl * S + cx) * 128);
                uint32_t h[4], l[4];
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(h[0]), "=r"(h[1]), "=r"(h[2]), "=r"(h[3]) : "r"(a));
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(l[0]), "=r"(l[1]), "=r"(l[2]), "=r"(l[3]) : "r"(a + T::PLANE_BYTES));
                float v[8];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 vh = um_h2f(h[j]), vl = um_h2f(l[j]);
                    v[2 * j]     = vh.x + vl.x;
                    v[2 * j + 1] = vh.y + vl.y;
                }
#pragma unroll
                for (int t = 0; t < T::TXT; ++t) {
                    const int kx = cx - t * S; // compile-time after unrolling
                    if (kx >= 0 && kx < 3) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc[t][j] = fmaf(wreg[ky * 3 + kx][j], v[j], acc[t][j]);
                    }
                }
            }
        }
        const int oy = ty * T::TH + tyl;
        if (oy < p.OH && c < p.Cp) {
#pragma unroll
            for (int t = 0; t < T::TXT; ++t) {
                const int ox = tx * T::TW + txl + t;
                if (ox < p.OW) {
                    float v[8];
                    if (fast_act) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = fminf(fmaxf(acc[t][j], acc[t][j] * slope), hi_clip);
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = umma_act(acc[t][j], p.act, p.alpha);
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = (c + j < p.C) ? v[j] : 0.0f; // channel padding stays zero
                    uint4 oh, ol;
                    um_split2(v[0], v[1], oh.x, ol.x);
                    um_split2(v[2], v[3], oh.y, ol.y);
                    um_split2(v[4], v[5], oh.z, ol.z);
                    um_split2(v[6], v[7], oh.w, ol.w);
                    const size_t o = (((size_t) n * p.OH + oy) * p.OW + ox) * p.Cp + c;
                    *reinterpret_cast<uint4*>(p.out_hi + o) = oh;
                    *reinterpret_cast<uint4*>(p.out_lo + o) = ol;
                }
            }
        }
        __syncthreads(); // everyone is done reading this stage
        if (tid == 0) {
            const int next = tile + DW_STAGES * gridDim.x;
            if (next < total) {
                fence_async_smem(); // generic-proxy reads above, async-proxy (TMA) writes below
                issue(next, stage);
            }
        }
    }
    (void) warp;
}

bool depthwise_tma_supported(const ConvArgs& a) {
    if (!a.in->lo || !a.out->lo) return false; // half-precision storage mode: the CUDA-core kernel (one plane)
    // tiles are 8x16 (stride 1) / 4x8 (stride 2) output pixels: tiny feature maps (7x7) would leave most of a tile empty
    const int tw = a.stride == 1 ? 16 : 8, th = a.stride == 1 ? 8 : 4;
    const int tx = (a.out->w + tw - 1) / tw, ty = (a.out->h + th - 1) / th;
    if ((double) a.out->w * a.out->h < 0.5 * (double) tx * tw * ty * th) return false;
    return a.k == 3 && (a.stride == 1 || a.stride == 2) && a.residual == nullptr && a.in->c == a.out->c && a.w->w_f32 != nullptr &&
           a.pad_mode <= SNNB_PAD_CONSTANT; // zero padding = the TMA out-of-bounds fill
}

template <int S> static int launch_depthwise_tma_s(snnb_context* ctx, const ConvArgs& a, EncodeTiledFn encode) {
    ctx->last_kernel = "depthwise_tma_kernel";
    using T = DwTile<S>;
    const snnb_tensor* in = a.in;
    snnb_tensor* out      = a.out;
    DwTmaParams p;
    p.out_hi = out->hi, p.out_lo = out->lo;
    p.w = a.w->w_f32, p.bias = a.w->bias;
    p.N = out->n, p.OH = out->h, p.OW = out->w, p.C = out->c, p.Cp = out->cp;
    p.pad_x = a.pad_x, p.pad_y = a.pad_y;
    p.tiles_x = (out->w + T::TW - 1) / T::TW, p.tiles_y = (out->h + T::TH - 1) / T::TH, p.chunks = (out->cp + 63) / 64;
    p.act = a.act, p.alpha = a.alpha;
    CUtensorMap tmI[2];
    {
        const cuuint64_t dims[4]    = {(cuuint64_t) in->c, (cuuint64_t) in->w, (cuuint64_t) in->h, (cuuint64_t) in->n}; // channels >= C read as zero
        const cuuint64_t strides[3] = {(cuuint64_t) in->cp * 2, (cuuint64_t) in->w * in->cp * 2, (cuuint64_t) in->h * in->w * in->cp * 2};
        const cuuint32_t box[4]     = {64, (cuuint32_t) T::IW, (cuuint32_t) T::IH, 1};
        const cuuint32_t estr[4]    = {1, 1, 1, 1};
        __half* planes[2]    = {in->hi, in->lo};
        for (int i = 0; i < 2; ++i) {
            CUresult r = encode(&tmI[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, planes[i], dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            SNNB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(depthwise input) failed: %d", (int) r);
        }
    }
    const uint32_t attr_bit = S == 1 ? ATTR_DW1 : ATTR_DW2;
    if (!(ctx->func_attr_mask & attr_bit)) {
        SNNB_CUDA_OK(cudaFuncSetAttribute(depthwise_tma_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_BYTES));
        ctx->func_attr_mask |= attr_bit;
    }
    const long long total = (long long) p.N * p.tiles_y * p.tiles_x * p.chunks;
    const int grid        = (int) std::min<long long>(total, 2 * ctx->sm_count); // two CTAs per SM (128 registers, <= 93 KB of shared memory each)
    const cudaError_t le  = launch_k_pdl(depthwise_tma_kernel<S>, dim3(grid), dim3(DW_THREADS), T::SMEM_BYTES, ctx->stream, tmI[0], tmI[1], p);
    cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("depthwise_tma_kernel launch failed: %s", cudaGetErrorString(e));
        return 1;
    }
    ctx->launches++;
    return 0;
}

int launch_depthwise_tma(snnb_context* ctx, const ConvArgs& a) {
    EncodeTiledFn encode = get_encode(ctx);
    SNNB_REQUIRE(encode, "launch_depthwise_tma: cuTensorMapEncodeTiled is unavailable in this driver");
    return a.stride == 1 ? launch_depthwise_tma_s<1>(ctx, a, encode) : launch_depthwise_tma_s<2>(ctx, a, encode);
}

// The stream-K schedule exactly as the kernel's roles derive it (decode_work / sk_first_work / sk_next_work run on the host here), one row
// {cta, tile, kb0, kb1, piece, pieces} per work item in each CTA's order: lets the CPU test suite check the integer arithmetic
// (coverage, piece numbering, balance) without a GPU. Returns the number of rows, or -1 when nothing would be cut.
int streamk_schedule(int tiles, int num_kb, int sms, int* rows, int capacity) {
    UmmaParams p {};
    int dp = 0, ctas = 0;
    long long units = 0;
    if (tiles <= 0 || num_kb <= 0 || sms <= 0 || tiles % sms == 0 || !streamk_split(tiles, num_kb, sms, dp, units, ctas)) return -1;
    p.sk = 1, p.sk_dp = dp, p.sk_ctas = ctas, p.sk_units = units, p.ksplit = 1, p.kb_per_split = num_kb;
    const int grid = dp > 0 ? sms : ctas, end = dp + 4 * ctas;
    int n = 0;
    for (int cta = 0; cta < grid; ++cta)
        for (int work = sk_first_work(p, cta, end); work < end; work = sk_next_work(p, work, cta, grid, num_kb, end)) {
            const WorkItem w = decode_work<true>(p, work, tiles, num_kb);
            if (n < capacity) {
                int* r = rows + 6 * (size_t) n;
                r[0] = cta, r[1] = w.tile, r[2] = w.kb0, r[3] = w.kb1, r[4] = w.piece, r[5] = w.pieces;
            }
            ++n;
        }
    return n;
}

// Every K block the producer loads, per work item, for a launch of `tiles` tiles with ksize x ksize taps over `cblocks` channel blocks
// (channel pitch icp) and a folded shortcut of sc_cblocks blocks: split-K into `ksplit` ranges, or stream-K over `sms` CTAs when
// ksplit == 0. The work items come from decode_work, the blocks from for_each_kblock - the functions the kernel's roles call. One row
// {tile, kb, sc, tap, cb, wcol} per K block. Returns the number of rows, or -1 for arguments no launch has (or nothing to cut for stream-K).
int kblock_schedule(int ksize, int cblocks, int icp, int sc_cblocks, int tiles, int ksplit, int sms, int* rows, int capacity) {
    if (ksize < 1 || cblocks < 1 || icp < 8 || sc_cblocks < 0 || tiles < 1 || ksplit < 0 || sms < 1) return -1;
    UmmaParams p {};
    p.ksize = ksize, p.cblocks = cblocks, p.ICp = icp, p.sc_cblocks = sc_cblocks, p.sc_stride = 1;
    const int num_kb = ksize * ksize * cblocks + sc_cblocks;
    std::vector<WorkItem> items;
    if (ksplit > 0) {
        p.ksplit = ksplit, p.kb_per_split = (num_kb + ksplit - 1) / ksplit;
        for (int work = 0; work < tiles * ksplit; ++work) items.push_back(decode_work<false>(p, work, tiles, num_kb));
    } else {
        int dp = 0, ctas = 0;
        long long units = 0;
        if (tiles % sms == 0 || !streamk_split(tiles, num_kb, sms, dp, units, ctas)) return -1;
        p.sk = 1, p.sk_dp = dp, p.sk_ctas = ctas, p.sk_units = units, p.ksplit = 1, p.kb_per_split = num_kb;
        const int grid = dp > 0 ? sms : ctas, end = dp + 4 * ctas;
        for (int cta = 0; cta < grid; ++cta)
            for (int work = sk_first_work(p, cta, end); work < end; work = sk_next_work(p, work, cta, grid, num_kb, end)) items.push_back(decode_work<true>(p, work, tiles, num_kb));
    }
    struct Row { // for_each_kblock is __host__ __device__: a functor with a callable of the same kind, not a host lambda
        int *rows, capacity, ksize, tile, n;
        __host__ __device__ void operator()(int kb, bool sc, int cb, int kx, int ky, int wcol) {
            if (n < capacity) {
                int* r = rows + 6 * (size_t) n;
                r[0] = tile, r[1] = kb, r[2] = sc, r[3] = ky * ksize + kx, r[4] = cb, r[5] = wcol;
            }
            ++n;
        }
    } row {rows, capacity, ksize, 0, 0};
    for (const WorkItem& w : items) {
        row.tile = w.tile;
        for_each_kblock(p, w.kb0, w.kb1, row);
    }
    return row.n;
}

} // namespace snnb

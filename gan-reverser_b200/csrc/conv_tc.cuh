// conv_tc.cuh -- implicit-GEMM convolution / linear layer on the 5th-gen tensor cores.
//
// One persistent kernel template serves every "real contraction" layer of G3 and R_default
// (models.lua:115-133, 414-451; SURVEY.md section 8a table "Implicit-GEMM view"):
//   D[128*MT pixels x NT channels] = sum over units (tap group g, 64-channel chunk cc), vertical
//   taps j < NDY:   A_{g,j,cc}[128 x 64] * W_{g,j,cc}[NT x 64]^T
//  * A tiles are boxes (64 ch, BW, BH+NDY-1, BN) of the NHWC bf16 activation fetched by TMA with
//    the tap offset added to the (w, h) coordinates; out-of-bounds rows are zero-filled by the
//    TMA unit, which *is* the conv's zero padding.  128B swizzle, K-major.
//  * HALO REUSE (NDY > 1): the NDY vertical taps of one horizontal offset read the same box
//    through UMMA descriptors offset by j*BW*128 bytes (a multiple of the 1024 B swizzle atom),
//    so a 3x3 conv ingests 3 boxes of BH+2 rows instead of 9 boxes of BH rows.
//  * RESIDENT WEIGHTS (BRES): when the layer's whole weight matrix fits in shared memory it is
//    loaded once per CTA and only activations stream.
//  * MT accumulators per CTA: every weight tile feeds MT MMAs (M = 128*MT per item).
//  * nearest-upsample + 3x3 conv (models.lua:121-122, 127-128) runs as four 2x2 phase
//    convolutions on the low-res input (weights pre-summed per phase at load time).
//  * tcgen05.mma (kind::f16, bf16 x bf16 -> fp32) is issued by one elected thread; accumulators
//    live in TMEM, double-buffered when 2*MT*NT <= 512 columns.  CG = 2: cta_group::2 CTA pairs
//    (M = 256 across the two SMs of a TPC, each CTA loads its own A tiles and half of every B
//    tile, only the leader issues; commits are multicast to both CTAs).
//  * epilogue: each warp loads TWO 32-column chunks per tcgen05.wait::ld, hands the accumulator
//    stage back to the MMA warp at once (registers are the third buffer), then folded-BN shift
//    (the BN scale is folded into the bf16 weights) -> ReLU/ELU/tanh/sigmoid -> optional 2x2
//    max-pool (warp shuffles) -> bf16 NHWC / fp32.  The chunk is staged in an XOR-swizzled smem
//    buffer that is TMA's 64B-swizzle layout: plain layers issue one cp.async.bulk.tensor store
//    per chunk, the others read it back for coalesced 16-byte st.global.cg.
//
// Why this shape (measured, DESIGN.md section 6): a B200 SM ingests ~128 B/clk through TMA with
// ~1300 cycles of latency, and the mbarrier round trip per pipeline stage costs 300+ cycles; a
// 128x128x64 MMA block needs 32 KB per 256 cycles, so without operand reuse inside the SM the
// tensor pipe idles.  Every knob above cuts ingested bytes per MMA-cycle.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one elected thread
// each), warps 2..9 = epilogue (two warps per TMEM lane quarter; warp 2 owns the TMEM
// allocation).  Only ONE lane ever polls an mbarrier: the other epilogue threads park on a
// hardware named barrier, because spinning try_waits measurably slow the TMA / MMA handshakes.
// Shape, activation, pooling, output type and CTA-pair mode are template parameters.
#pragma once
#include "common.cuh"

#ifndef GANREV_STORE_EARLY
#define GANREV_STORE_EARLY 1
#endif
#ifndef GANREV_POOL_DIRECT
#define GANREV_POOL_DIRECT 1
#endif

namespace ganrev {
namespace tc {

constexpr int kEpiWarps = 8;                 // two warps per TMEM lane quarter; (sub-tile, column chunk) pairs round-robin
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                  // bf16 elements = 128 bytes = one swizzle span
constexpr int kMaxStages = 8;
constexpr int kSmemBudget = 227 * 1024;
constexpr unsigned long long kSpinLimitCycles = 4000000000ull;  // ~2 s: turn a hang into a trap

template <int NT, int MT, int CG = 1> struct Cfg {
    static constexpr int kBBytes = (NT / CG) * kBlockK * 2;             // this CTA's share of one 64-wide weight tile
    static constexpr int kNAcc = (2 * MT * NT <= 512) ? 2 : 1;          // accumulator buffers
    static constexpr int kCols = kNAcc * MT * NT;
    static constexpr int kTmemCols = kCols <= 32 ? 32 : (kCols <= 64 ? 64 : (kCols <= 128 ? 128 : (kCols <= 256 ? 256 : 512)));
    static constexpr int kChunk = NT < 32 ? NT : 32;                    // accumulator columns per tcgen05.ld
    static constexpr int kBarBytes = (2 * kMaxStages + 5) * 8 + 24;     // full/empty per stage, tfull/tempty x2, bres, tmem slot (16 B aligned)
    static constexpr int kXposeOff = (kBarBytes + 2 * NT * 4 + 1023) / 1024 * 1024;   // store buffers start on a swizzle-pattern boundary (TMA store)
    static constexpr int kSsBytes = 2 * NT * 4;                         // double-buffered shift
    static constexpr int kXposeBytes = kEpiWarps * 32 * 64;             // per-warp 32 px x 64 B store-transpose buffers
};

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as an error, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err_flag, int code) {
    if (mbar_try_wait(bar, parity)) return;
    const unsigned long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > kSpinLimitCycles) {
            if (err_flag) atomicExch(err_flag, code);
            __threadfence_system();
            __trap();
        }
    }
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// TMA store of one 4-D box from shared memory (bulk async-group completion)
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }   // all but the latest store have read their source
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---- cta_group::2 (CTA pair on one TPC): one MMA spans both SMs (M = 256); each SM supplies its own
// 128 rows of A and HALF of the B tile, so the per-SM shared-memory operand reads per MMA drop.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-rank bit: "the leader CTA's copy of this barrier"
__device__ __forceinline__ void tma_load_4d_cg2(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_cg2(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint32_t bar, uint32_t cta) {   // arrive on the same barrier in CTA `cta` of the cluster
    asm volatile(
        "{\n\t.reg .b32 remAddr32;\n\t"
        "mapa.shared::cluster.u32 remAddr32, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [remAddr32];\n\t}"
        ::"r"(bar), "r"(cta) : "memory");
}
__device__ __forceinline__ void umma_bf16_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_cg2(uint32_t bar) {   // arrives on `bar` in BOTH CTAs of the pair
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}
template <int COLS> __device__ __forceinline__ void tmem_alloc_cg2(uint32_t dst_smem) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS> __device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}

template <int COLS> __device__ __forceinline__ void tmem_alloc(uint32_t dst_smem) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS> __device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; one elected thread issues this for the whole CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once every previously issued tcgen05 op of this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i = lane base+i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row atoms of 1024 B (SBO), sm_100
// descriptor version 1.  (cute/arch/mma_sm100_desc.hpp SmemDescriptor bit layout.)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);        // [0,14)  start address >> 4
    d |= static_cast<uint64_t>(0) << 16;                         // [16,30) LBO (unused for swizzled K-major)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;                 // [32,46) SBO = 1024 B
    d |= static_cast<uint64_t>(1) << 46;                         // [46,48) version = 1 (sm_100)
    d |= static_cast<uint64_t>(2) << 61;                         // [61,64) SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=NT.
template <int NT, int M = kBlockM> __device__ __forceinline__ constexpr uint32_t make_idesc() {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(NT >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

constexpr int ACT_RUNTIME = -1;
template <int ACT> __device__ __forceinline__ float act_fn(float v, int runtime_act) {
    if (ACT == ACT_RELU) return fmaxf(v, 0.0f);
    if (ACT == ACT_ELU) return elu_fast(v);
    if (ACT == ACT_NONE) return v;
    if (ACT == ACT_SIGMOID) return __fdividef(1.0f, 1.0f + __expf(-v));
    return apply_act(v, runtime_act);
}
// Warp-uniform leader election: keeps the issuing code convergent so TMA / tcgen05 instructions
// (which take uniform registers) compile to straight-line code instead of per-thread loops.
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// debug timeline: role r, event e -> clock64 of CTA 0
#ifndef GANREV_EPI_TRACE
#define GANREV_TR(role, e)                                                                     \
    do {                                                                                       \
        if (p.trace != nullptr && blockIdx.x == 0 && (e) < 256) p.trace[(role) * 256 + (e)] = clock64(); \
    } while (0)
#define GANREV_TRE(role, e) do {} while (0)
#else   // -DGANREV_EPI_TRACE: rows 0..3 hold the phases of epilogue thread 0's chunks instead of the producer / MMA events
#define GANREV_TR(role, e)                                                                     \
    do {                                                                                       \
        if ((role) >= 4 && p.trace != nullptr && blockIdx.x == 0 && (e) < 256) p.trace[(role) * 256 + (e)] = clock64(); \
    } while (0)
#define GANREV_TRE(role, e)                                                                    \
    do {                                                                                       \
        if (etid == 0 && p.trace != nullptr && blockIdx.x == 0 && (e) < 256) p.trace[(role) * 256 + (e)] = clock64(); \
    } while (0)
#endif

// M-tile index -> first image / row / column of the tile
struct TileCoord {
    int n0, h0, w0;
};
__device__ __forceinline__ TileCoord decode_tile(const ConvGemm& p, int tile) {
    TileCoord c;
    c.w0 = (tile & (p.tiles_w - 1)) << p.lgBW;      // tiles_w, tiles_h are powers of two
    const int t = tile >> p.lgTW;
    c.h0 = (t & (p.tiles_h - 1)) << p.lgBH;
    c.n0 = (t >> p.lgTH) << p.lgBN;
    return c;
}
// item -> (M group, phase, N tile); N tile fastest so consecutive items share activations in L2
struct ItemCoord {
    int mgroup, phase, ntile;
};
__device__ __forceinline__ ItemCoord decode_item(const ConvGemm& p, int item) {
    ItemCoord c;
    int t;
    if (p.lgNT >= 0) { c.ntile = item & (p.n_tiles - 1); t = item >> p.lgNT; }
    else             { t = item / p.n_tiles; c.ntile = item - t * p.n_tiles; }
    c.phase = p.nphase == 4 ? (t & 3) : 0;          // nphase is 1 or 4
    c.mgroup = p.nphase == 4 ? (t >> 2) : t;
    return c;
}

// two fp32 FMAs per instruction (FFMA2): the fused tap products below are bound by issue slots, not by the FMA pipe
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ unsigned long long pack_f32x2(float lo, float hi) {
    unsigned long long d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}

// FUSE3 = C (G's Up+Conv 256->128 + BN + ReLU, models.lua:127-130): the layer's activation is consumed where it is
// produced.  The last conv (128 -> C, 3x3, models.lua:132) needs, per pixel, the 9*C products <act[pixel][0..127], w3[tap][co]>;
// each epilogue warp owns one 128-pixel sub-tile (lane = pixel, all 128 channels in two rounds of two 32-column chunks),
// keeps 9*C packed (even, odd channel) fp32 sums per thread and writes them as planes P[tap*C + co][pixel] -- 36*C B per pixel
// instead of the 256 B bf16 activation, and the separate tap-product GEMM (a full HBM round trip of that activation)
// disappears.  The weights sit in shared memory as fp32 (16-byte broadcast loads); the activation is NOT rounded to bf16.
// MASKSUM (G's backward convs conv2^T / conv1^T, refinement): the pooled epilogue SUMS the 2x2 window (the adjoint of nearest
// upsampling) and multiplies by [ref > 0], the stored forward activation (the ReLU mask) -- ref has the output's NHWC layout,
// so each lane loads its 16 bytes of ref at the offset it stores to.  No shift, no activation.
template <int NT, int MT, int NDY, bool BRES, int ACT, bool POOL, bool OUT_FP32, int CG, int FUSE3 = 0, bool MASKSUM = false>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmO, const __grid_constant__ ConvGemm p, const int n_items) {
    using C = Cfg<NT, MT, CG>;
    constexpr int NACC = C::kNAcc;
    // Programmatic dependent launch: the NEXT kernel of the stream may become resident as soon as this grid's CTAs leave their SMs
    // (its barrier init / TMEM allocation / descriptor prefetch / resident-weight loads then overlap this grid's tail); it waits
    // for this grid's completion itself (griddepcontrol.wait below) before it touches an activation.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;          // CG == 2: rank 0 is the leader (issues the MMAs)
    const int unit0 = static_cast<int>(blockIdx.x) / CG;             // persistent loop over items, one CTA pair (or CTA) each
    const int ustep = static_cast<int>(gridDim.x) / CG;
    extern __shared__ uint8_t smem_raw[];
    // 128B swizzle needs 1024 B alignment of every operand tile
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (smem_base - smem_u32(smem_raw));
    const int S = p.stages;
    const int kb_total = p.units * NDY;                                   // k-blocks per item
    const uint32_t bres_bytes = BRES ? static_cast<uint32_t>(kb_total) * C::kBBytes : 0u;
    const uint32_t stage0 = smem_base + bres_bytes;                       // resident weights first, then the ring
    const uint32_t tail_off = bres_bytes + static_cast<uint32_t>(S) * p.stage_bytes;
    const uint32_t bar_base = smem_base + tail_off;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (kMaxStages + s); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kMaxStages + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kMaxStages + 2 + a); };
    const uint32_t bres_bar = bar_base + 8u * (2 * kMaxStages + 4);
    const uint32_t tmem_slot = bar_base + 8u * (2 * kMaxStages + 5);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + tail_off + 8 * (2 * kMaxStages + 5));

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full_bar(s), CG);                // CG == 2: the leader's copy collects both producers
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull_bar(a), 1);
            mbar_init(tempty_bar(a), CG * kEpiWarps);  // one arrival per epilogue warp (of both CTAs, on the leader)
        }
        mbar_init(bres_bar, 1);
        fence_barrier_init();
    }
    if (warp == 2) { if (CG == 2) tmem_alloc_cg2<C::kTmemCols>(tmem_slot); else tmem_alloc<C::kTmemCols>(tmem_slot); }
    tcgen05_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (BRES && CG == 2) {
        // Resident weights of BOTH CTAs must be in place before the leader issues an MMA that reads
        // the peer's half: each CTA loads its rows, one thread waits, then the pair synchronises.
        if (warp == 0 && elect_one_sync()) {
            mbar_expect_tx(bres_bar, bres_bytes);
            for (int kb = 0; kb < kb_total; ++kb)
                tma_load_2d(smem_base + kb * C::kBBytes, &tmB, bres_bar, kb * kBlockK, static_cast<int>(rank) * (NT / CG));
        }
        if (threadIdx.x == 32) mbar_wait(bres_bar, 0u, p.err_flag, 105);
        cluster_sync_all();
    }

    // everything above touched only this kernel's own shared memory / TMEM and the (constant) weights; from here on the producer
    // reads the previous kernel's output and the epilogue overwrites what the previous kernel may still be reading
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer (one elected thread)
        if (elect_one_sync()) {
            if (BRES && CG == 1) {   // the whole weight matrix of this layer, once (nphase == n_tiles == 1)
                mbar_expect_tx(bres_bar, bres_bytes);
                for (int kb = 0; kb < kb_total; ++kb)
                    tma_load_2d(smem_base + kb * C::kBBytes, &tmB, bres_bar, kb * kBlockK, static_cast<int>(rank) * (NT / CG));
            }
            int stage = 0, tr_p = 0;
            uint32_t phase = 0;
            const uint32_t unit_tx = ((p.dbg & 1) ? 0u : static_cast<uint32_t>(MT * p.a_unit_bytes)) +
                                     ((BRES || (p.dbg & 2)) ? 0u : static_cast<uint32_t>(NDY * C::kBBytes));
            for (int item = unit0; item < n_items; item += ustep) {
                const ItemCoord c = decode_item(p, item);
                const int brow = c.phase * p.cout_pad + c.ntile * NT + static_cast<int>(rank) * (NT / CG);
                TileCoord tc[MT];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) tc[mt] = decode_tile(p, (c.mgroup * CG + static_cast<int>(rank)) * MT + mt);   // tiles past the end read OOB zeros
                int g = 0, cc = 0;
                for (int u0 = 0; u0 < p.units; u0 += p.ups) {
                    const int nu = min(p.ups, p.units - u0);
                    mbar_wait(empty_bar(stage), phase ^ 1u, p.err_flag, 101);
                    GANREV_TR(0, tr_p);
                    const uint32_t s_base = stage0 + stage * p.stage_bytes;
                    if (CG == 1 || rank == 0) mbar_expect_tx(full_bar(stage), nu * unit_tx * CG);   // bytes of both CTAs land on the leader's barrier
                    else mbar_arrive_cta(full_bar(stage), 0);
                    for (int x = 0; x < nu; ++x) {
                        const uint32_t u_base = s_base + x * p.unit_bytes;
                        const int dx = p.gdx[c.phase][g], dy = p.gdy0[c.phase][g];
                        if (!(p.dbg & 1)) {
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt) {
                                if (CG == 2) tma_load_4d_cg2(u_base + mt * p.a_unit_bytes, &tmA, full_bar(stage), cc * kBlockK, tc[mt].w0 + dx, tc[mt].h0 + dy, tc[mt].n0);
                                else tma_load_4d(u_base + mt * p.a_unit_bytes, &tmA, full_bar(stage), cc * kBlockK, tc[mt].w0 + dx, tc[mt].h0 + dy, tc[mt].n0);
                            }
                        }
                        if (!BRES && !(p.dbg & 2)) {
#pragma unroll
                            for (int j = 0; j < NDY; ++j) {
                                if (CG == 2) tma_load_2d_cg2(u_base + MT * p.a_unit_bytes + j * C::kBBytes, &tmB, full_bar(stage), (g * NDY + j) * p.Cin + cc * kBlockK, brow);
                                else tma_load_2d(u_base + MT * p.a_unit_bytes + j * C::kBBytes, &tmB, full_bar(stage), (g * NDY + j) * p.Cin + cc * kBlockK, brow);
                            }
                        }
                        if (++cc == p.cin_chunks) { cc = 0; ++g; }
                    }
                    GANREV_TR(1, tr_p);
                    ++tr_p;
                    if (++stage == S) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (one elected thread; CG == 2: leader CTA only)
        if (rank == 0 && elect_one_sync()) {
            constexpr uint32_t idesc = make_idesc<NT, kBlockM * CG>();
            const uint64_t desc_base = make_smem_desc(0);
            auto desc_at = [&](uint32_t addr) { return desc_base | static_cast<uint64_t>((addr & 0x3FFFFu) >> 4); };
            if (BRES && CG == 1) {                   // (CG == 2: both CTAs' resident weights were awaited before the cluster sync below)
                mbar_wait(bres_bar, 0u, p.err_flag, 105);
                tcgen05_fence_after();
            }
            int stage = 0, tr_m = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int item = unit0; item < n_items; item += ustep, ++it) {
                const int acc = it % NACC;
                const uint32_t acc_phase = (it / NACC) & 1u;
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u, p.err_flag, 102);
                GANREV_TR(6, it);
                tcgen05_fence_after();
                int g = 0, cc = 0;
                for (int u0 = 0; u0 < p.units; u0 += p.ups) {
                    const int nu = min(p.ups, p.units - u0);
                    mbar_wait(full_bar(stage), phase, p.err_flag, 103);
                    GANREV_TR(2, tr_m);
                    tcgen05_fence_after();
                    const uint32_t s_base = stage0 + stage * p.stage_bytes;
                    for (int x = 0; x < nu; ++x) {
                        const uint32_t u_base = s_base + x * p.unit_bytes;
                        const uint32_t b_base = BRES ? smem_base + ((g * NDY) * p.cin_chunks + cc) * C::kBBytes
                                                     : u_base + MT * p.a_unit_bytes;
                        const uint32_t b_step = BRES ? static_cast<uint32_t>(p.cin_chunks) * C::kBBytes : static_cast<uint32_t>(C::kBBytes);
                        if (!(p.dbg & 8)) {
#pragma unroll
                            for (int j = 0; j < NDY; ++j) {
                                const uint64_t bdesc = desc_at(b_base + j * b_step);
#pragma unroll
                                for (int mt = 0; mt < MT; ++mt) {
                                    // vertical tap j = the same box, j*BW rows (a multiple of the 1024 B atom) further down
                                    const uint64_t adesc = desc_at(u_base + mt * p.a_unit_bytes + j * p.dy_stride_bytes);
                                    const uint32_t tmem_d = tmem_base + static_cast<uint32_t>((acc * MT + mt) * NT);
                                    const bool first = (u0 + x == 0) && (j == 0);
#pragma unroll
                                    for (int k = 0; k < kBlockK / 16; ++k) {   // +32 B per K=16 step inside the swizzle span (>>4 -> +2)
                                        if (CG == 2) umma_bf16_cg2(tmem_d, adesc + 2u * k, bdesc + 2u * k, idesc, (first && k == 0) ? 0u : 1u);
                                        else umma_bf16(tmem_d, adesc + 2u * k, bdesc + 2u * k, idesc, (first && k == 0) ? 0u : 1u);
                                    }
                                }
                            }
                        }
                        if (++cc == p.cin_chunks) { cc = 0; ++g; }
                    }
                    if (CG == 2) {
                        umma_commit_cg2(empty_bar(stage));                          // frees the slot in BOTH CTAs when the MMAs retire
                        if (u0 + p.ups >= p.units) umma_commit_cg2(tfull_bar(acc)); // accumulators complete (both CTAs' epilogues)
                    } else {
                        umma_commit(empty_bar(stage));                              // frees the smem slot when the MMAs retire
                        if (u0 + p.ups >= p.units) umma_commit(tfull_bar(acc));     // accumulators complete
                    }
                    GANREV_TR(3, tr_m);
                    ++tr_m;
                    if (++stage == S) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..9)
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int sub = (warp - 2) >> 2;        // which (sub-tile, chunk) pairs this warp takes
        const int etid = threadIdx.x - 64;      // 0..255
        const int m = q * 32 + lane;            // tile row = pixel
        const int BW = 1 << p.lgBW;
        const int w_l = m & (BW - 1);
        const int h_l = (m >> p.lgBW) & ((1 << p.lgBH) - 1);
        const int n_l = m >> (p.lgBW + p.lgBH);
        // pooled TMA store: this lane's slot among the quarter's (bw/2) x (bh/2) pooled pixels (bw = min(BW, 32) columns per quarter row)
        const int lg_bw = min(p.lgBW, 5);
        const bool pool_writer = !(w_l & 1) && !(h_l & 1);
        const int pool_row = ((lane >> lg_bw) >> 1) * ((1 << lg_bw) >> 1) + ((lane & ((1 << lg_bw) - 1)) >> 1);
        const int qw0 = (q * 32) & (BW - 1), qh0 = ((q * 32) >> p.lgBW) & ((1 << p.lgBH) - 1), qn0 = (q * 32) >> (p.lgBW + p.lgBH);   // first pixel of this warp's lane quarter
        float* ss_base = reinterpret_cast<float*>(smem + tail_off + C::kBarBytes);
        // 2 KB per warp and buffer; xpose2: two buffers per warp, alternating per TMA store
        uint4* const xpose0 = reinterpret_cast<uint4*>(smem + tail_off + C::kXposeOff) + (warp - 2) * 128 * (p.xpose2 ? 2 : 1);
        int xcur = 0;
        constexpr int CW = C::kChunk;
        constexpr int kChunksPerTile = NT / CW;
        constexpr int kPairs = MT * kChunksPerTile;           // (sub-tile, column chunk) pairs per item
        constexpr int kStep = kEpiWarps / 4;                  // warps per TMEM lane quarter
        constexpr int kIters = (kPairs + kStep - 1) / kStep;  // pairs per warp
        static_assert(kPairs % kStep == 0 || kIters == 1, "pairs must split evenly over the warps of a quarter");
        static_assert(MT == 1 || kChunksPerTile % kStep == 0, "a warp's sub-tile index must be a compile-time constant");
        constexpr bool kRec = OUT_FP32 && (NT == 16 || NT == 32);   // fp32 records of 16 / 32 floats per pixel (G conv3 pass 1)
        // transposed (coalesced) store path: bf16 NHWC, or the fp32 tap records
        const bool xposed = !OUT_FP32 || (kRec && p.out_sC == 1 && p.out_sP == NT);
        const bool run = !(p.dbg & 4) && sub < kPairs;
        const bool no_store = (p.dbg & 16) != 0;
        const int jj = lane & 3;
        constexpr int kTaps = 9 * FUSE3;
        // plain bf16 layers (the TMA-store epilogue): per round math A, store A, math B, store B, so that A's bulk store has read its
        // staging buffer by the time B needs it (the ELU math of a chunk is MUFU-bound, interleaving two chunks buys nothing there);
        // the pooled / fp32 layers keep both chunks' math in one basic block
        // (measured, same box: R conv2 7.62 -> 7.13 ms, R conv4 3.28 -> 2.98 ms per 32768 faces; G's Linear, which has two staging
        // buffers and cheap ReLU math, is 7 % faster with the interleaved order and keeps it)
        // pooled bf16 layers: the four lanes of a 2x2 window split the chunk's 32 channels between them WHILE pooling (each exchange
        // keeps half of the channels: 24 shuffles instead of 64), so each lane ends with 8 pooled channels: shift + ELU on 8 values
        // instead of 32 (the pooled epilogue was bound by 32 ex2 per lane and chunk of which 24 were thrown away) and one 16-byte
        // st.global per lane -- a window's four lanes write its 64 contiguous bytes, no shared-memory transpose
        constexpr bool kPoolDirect = GANREV_POOL_DIRECT && POOL && !OUT_FP32 && C::kChunk == 32;
        constexpr bool kStoreEarly = GANREV_STORE_EARLY && !POOL && !OUT_FP32 && ACT == ACT_ELU;
        static_assert(!MASKSUM || (kPoolDirect && FUSE3 == 0), "MASKSUM is a mode of the direct pooled epilogue");
        if constexpr (FUSE3 != 0) {   // tap weights of the last conv -> shared memory (the store-transpose buffers are unused here)
            static_assert(NT == 128 && MT == 2 && !POOL && !OUT_FP32 && ACT == ACT_RELU && kEpiWarps == 8, "FUSE3 is G's Up+Conv 256->128");
            static_assert(kTaps * 128 * 4 <= C::kXposeBytes, "tap weights must fit in the store-transpose buffers");
            float* w3s = reinterpret_cast<float*>(smem + tail_off + C::kXposeOff);
            for (int i = etid; i < kTaps * 128; i += 32 * kEpiWarps) w3s[i] = __ldg(p.w3 + i);
            named_bar_sync(1, 32 * kEpiWarps);
        }
        int it = 0;
        for (int item = unit0; item < n_items; item += ustep, ++it) {
            const ItemCoord c = decode_item(p, item);
            const int acc = it % NACC;
            const uint32_t acc_phase = (it / NACC) & 1u;
            const int cbase = c.ntile * NT;
            // stage this item's folded-BN shift (double-buffered; the named barrier of item
            // i+1 proves every warp is done reading the buffer of item i).  Layers with a single
            // N tile keep one copy for the whole kernel.
            float* ss = ss_base + (p.n_tiles > 1 ? (it & 1) * NT : 0);
            if (p.n_tiles > 1 || it == 0) {
                for (int i = etid; i < NT; i += 32 * kEpiWarps) ss[i] = __ldg(p.shift + cbase + i);
                named_bar_sync(1, 32 * kEpiWarps);
            }
            if constexpr (FUSE3 != 0) {
                // warp (q, sub) owns sub-tile `sub`: lane = pixel, 4 chunks of 32 channels in two rounds
                const TileCoord t = decode_tile(p, (c.mgroup * CG + static_cast<int>(rank)) * MT + sub);
                const int n = t.n0 + n_l, oh = 2 * (t.h0 + h_l) + (c.phase >> 1), ow = 2 * (t.w0 + w_l) + (c.phase & 1);
                const bool wr = n < p.n_img && !no_store;
                float* dst = p.taps + (static_cast<long long>(n) * p.Hout + oh) * p.Wout + ow;
                const ulonglong2* w3v = reinterpret_cast<const ulonglong2*>(smem + tail_off + C::kXposeOff);   // [9*C][32] x 4 channels
                if (etid == 0) {
                    GANREV_TR(7, it);
                    mbar_wait(tfull_bar(acc), acc_phase, p.err_flag, 104);   // the only poller
                    GANREV_TR(4, it);
                }
                named_bar_sync(2, 32 * kEpiWarps);
                tcgen05_fence_after();
                const uint32_t tq = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * MT + sub) * NT);
                unsigned long long s9[kTaps];
#pragma unroll
                for (int tp = 0; tp < kTaps; ++tp) s9[tp] = 0ull;
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    uint32_t ra[32], rb[32];
                    tmem_ld32(tq + (2 * r) * 32, ra);
                    tmem_ld32(tq + (2 * r + 1) * 32, rb);
                    tmem_ld_wait();
                    if (r == 1) {   // the registers are the third buffer: hand the accumulator stage back at once
                        tcgen05_fence_before();
                        __syncwarp();
                        if (lane == 0) { if (CG == 2) mbar_arrive_cta(tempty_bar(acc), 0); else mbar_arrive(tempty_bar(acc)); }
                    }
                    if (!(p.dbg & 4)) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {     // channels 64*r + 4*j .. +3
                            const float4 sh = *reinterpret_cast<const float4*>(ss + 64 * r + 4 * j);
                            const uint32_t* a = j < 8 ? &ra[4 * j] : &rb[4 * (j - 8)];
                            const unsigned long long v01 = pack_f32x2(fmaxf(__uint_as_float(a[0]) + sh.x, 0.0f), fmaxf(__uint_as_float(a[1]) + sh.y, 0.0f));
                            const unsigned long long v23 = pack_f32x2(fmaxf(__uint_as_float(a[2]) + sh.z, 0.0f), fmaxf(__uint_as_float(a[3]) + sh.w, 0.0f));
#pragma unroll
                            for (int tp = 0; tp < kTaps; ++tp) {
                                const ulonglong2 w = w3v[tp * 32 + 16 * r + j];
                                s9[tp] = ffma2(v01, w.x, s9[tp]);
                                s9[tp] = ffma2(v23, w.y, s9[tp]);
                            }
                        }
                    }
                }
                if (wr) {
#pragma unroll
                    for (int tp = 0; tp < kTaps; ++tp)
                        __stcg(dst + tp * p.taps_plane, __uint_as_float(static_cast<uint32_t>(s9[tp])) + __uint_as_float(static_cast<uint32_t>(s9[tp] >> 32)));
                }
                if (etid == 0) GANREV_TR(5, it);
            } else {
            // Output offsets of this item's tiles, computed while the MMAs are still running.
            // offs[mt][i]: element offset of pixel (lane>>2) + 8*i of this warp's quarter (the pixel a
            // group of 4 lanes stores after the transpose), -1 = nothing to store.
            long long offs[MT][4];
            size_t pix_off[MT];
            bool writer[MT], live[MT];
            TileCoord tco[MT];
            const bool by_tma = !OUT_FP32 && !kPoolDirect && p.tma_store && !p.tma_hybrid;   // TMA stores address by tile coordinates: no per-pixel offsets needed
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const TileCoord t = decode_tile(p, (c.mgroup * CG + static_cast<int>(rank)) * MT + mt);
                tco[mt] = t;
                live[mt] = false;
                if (by_tma) {
                    pix_off[mt] = 0; writer[mt] = false;
#pragma unroll
                    for (int i = 0; i < 4; ++i) offs[mt][i] = -1ll;
                    continue;
                }
                const int n = t.n0 + n_l, h = t.h0 + h_l, w = t.w0 + w_l;
                int oh = h, ow = w;
                writer[mt] = n < p.n_img;
                live[mt] = writer[mt] && !no_store;
                if (POOL) {
                    oh = h >> 1; ow = w >> 1;
                    writer[mt] = writer[mt] && !(h & 1) && !(w & 1);
                } else if (p.up == 2) {
                    oh = 2 * h + (c.phase >> 1); ow = 2 * w + (c.phase & 1);
                }
                pix_off[mt] = static_cast<size_t>(n) * p.out_sN + (static_cast<size_t>(oh) * p.Wout + ow) * p.out_sP;
                const long long my_off = (writer[mt] && !no_store) ? static_cast<long long>(pix_off[mt]) : -1ll;
#pragma unroll
                for (int i = 0; i < 4; ++i) offs[mt][i] = (xposed && !kPoolDirect) ? __shfl_sync(0xffffffffu, my_off, (lane >> 2) + 8 * i) : -1ll;
            }
            if (etid == 0) {
                GANREV_TR(7, it);
                mbar_wait(tfull_bar(acc), acc_phase, p.err_flag, 104);   // the only poller
                GANREV_TR(4, it);
            }
            named_bar_sync(2, 32 * kEpiWarps);
            tcgen05_fence_after();
            const uint32_t tq_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * MT * NT);

            // accumulator columns -> shift, pool, activation (registers only; two of these back to
            // back form one basic block, so the compiler interleaves their dependency chains)
            auto math = [&](const int pair, const uint32_t (&a)[32], float (&v)[32]) {
                const int c0 = (pair % kChunksPerTile) * CW;
#pragma unroll
                for (int j = 0; j < CW / 4; ++j) {   // folded-BN shift (the scale lives in the weights)
                    const float4 sh = *reinterpret_cast<const float4*>(ss + c0 + 4 * j);
                    v[4 * j + 0] = __uint_as_float(a[4 * j + 0]) + sh.x;
                    v[4 * j + 1] = __uint_as_float(a[4 * j + 1]) + sh.y;
                    v[4 * j + 2] = __uint_as_float(a[4 * j + 2]) + sh.z;
                    v[4 * j + 3] = __uint_as_float(a[4 * j + 3]) + sh.w;
                }
                if (POOL) {
                    // 2x2 max: w-neighbour is lane^1, h-neighbour is lane^BW (BW <= 16)
#pragma unroll
                    for (int j = 0; j < CW; ++j) {
                        v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 1));
                        v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], BW));
                    }
                }
#pragma unroll
                for (int j = 0; j < CW; ++j) v[j] = act_fn<ACT>(v[j], p.act);
            };
            auto store = [&](const int pair, const int mt, const float (&v)[32], const bool use_tma) {
                const int c0 = (pair % kChunksPerTile) * CW;
                long long o4[4] = {-1, -1, -1, -1};
                size_t po = 0;
                bool wr = false;
                TileCoord tt = tco[0];
#pragma unroll
                for (int m2 = 0; m2 < MT; ++m2)
                    if (m2 == mt) {
                        po = pix_off[m2]; wr = writer[m2]; tt = tco[m2];
#pragma unroll
                        for (int i = 0; i < 4; ++i) o4[i] = offs[m2][i];
                    }
                if (xposed) {
                    // Each lane owns one pixel's 64 B of this chunk (32 bf16 channels, or 16 floats of
                    // the G conv3 tap record; 32-float records take two passes).  Transpose through an
                    // XOR-swizzled smem buffer so 4 lanes store one pixel's contiguous 64 B (8 pixels
                    // per instruction) instead of 32 lanes hitting 32 different lines.
                    constexpr int kPasses = (OUT_FP32 && NT == 32) ? 2 : 1;
#pragma unroll
                    for (int hpass = 0; hpass < kPasses; ++hpass) {
                        uint4* const xpose = xpose0 + xcur * 128;
                        if (!OUT_FP32 && p.tma_store) { if (p.xpose2) tma_store_wait_read1(); else tma_store_wait_read(); }   // the store that last used this buffer has read it (no-op when none is pending)
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            uint4 pk;
                            if (OUT_FP32) {
                                const int b0 = 16 * hpass + 4 * j;
                                pk = make_uint4(__float_as_uint(v[b0]), __float_as_uint(v[b0 + 1]), __float_as_uint(v[b0 + 2]), __float_as_uint(v[b0 + 3]));
                            } else {
                                pk.x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
                                pk.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
                                pk.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
                                pk.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
                            }
                            if (POOL && !OUT_FP32 && use_tma) {   // pooled: only the even-(h, w) lanes hold a result; pack them densely
                                if (pool_writer) xpose[pool_row * 4 + (j ^ ((pool_row >> 1) & 3))] = pk;
                            } else {
                                xpose[lane * 4 + (j ^ ((lane >> 1) & 3))] = pk;
                            }
                        }
                        if (!OUT_FP32 && use_tma) {
                            // The buffer is exactly a [32 pixels][32 channels] bf16 box in TMA's 64B-swizzle layout: one
                            // bulk tensor store per chunk replaces the read-back, the address math and the predicated STGs
                            // (pixels past the end of the batch are clipped by the tensor map).
                            fence_proxy_async_smem();
                            __syncwarp();
                            if (lane == 0 && !no_store) {
                                if (POOL) tma_store_4d(&tmO, smem_u32(xpose), cbase + c0, (tt.w0 + qw0) >> 1, (tt.h0 + qh0) >> 1, tt.n0 + qn0);
                                else tma_store_4d(&tmO, smem_u32(xpose), cbase + c0, tt.w0 + qw0, tt.h0 + qh0, tt.n0 + qn0);
                            }
                            if (p.xpose2) xcur ^= 1;
                            continue;
                        }
                        __syncwarp();
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int px = (lane >> 2) + 8 * i;
                            const uint4 val = xpose[px * 4 + (jj ^ ((px >> 1) & 3))];
                            if (o4[i] >= 0) {
                                // st.global.cg: activations are consumed by the NEXT kernel, never re-read here
                                if (OUT_FP32) __stcg(reinterpret_cast<uint4*>(reinterpret_cast<float*>(p.out) + o4[i] + 16 * hpass + jj * 4), val);
                                else __stcg(reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.out) + o4[i] + cbase + c0 + jj * 8), val);
                            }
                        }
                    }
                } else if (OUT_FP32) {
                    if (wr && !no_store) {
                        float* o = reinterpret_cast<float*>(p.out) + po + static_cast<size_t>(cbase + c0) * p.out_sC;
#pragma unroll
                        for (int j = 0; j < CW; ++j)
                            if (cbase + c0 + j < p.cout_real) o[static_cast<size_t>(j) * p.out_sC] = v[j];
                    }
                }
            };
            // Two pairs per round: both tcgen05.ld are issued together and awaited once, then the
            // math of both runs as one instruction stream.  After the LAST load has landed the
            // accumulator stage is handed back to the MMA warp at once -- the registers are the
            // third buffer, so the tensor pipe never waits for activation math or stores.
            if (run) {
#pragma unroll
                for (int i0 = 0; i0 < kIters; i0 += 2) {
                    const bool two = i0 + 1 < kIters;
                    const int pa = sub + i0 * kStep, pb = pa + kStep;
                    // kChunksPerTile is a multiple of kStep (or MT == 1), so the sub-tile is known at compile time
                    const int mta = (i0 * kStep) / kChunksPerTile, mtb = ((i0 + 1) * kStep) / kChunksPerTile;
                    uint32_t ra[32], rb[32];
                    if (CW == 32) tmem_ld32(tq_base + pa * CW, ra); else tmem_ld16(tq_base + pa * CW, ra);
                    if (two) { if (CW == 32) tmem_ld32(tq_base + pb * CW, rb); else tmem_ld16(tq_base + pb * CW, rb); }
                    tmem_ld_wait();
                    GANREV_TRE(0, it * 4 + i0);
                    if (i0 + 2 >= kIters) {
                        tcgen05_fence_before();
                        __syncwarp();
                        if (lane == 0) { if (CG == 2) mbar_arrive_cta(tempty_bar(acc), 0); else mbar_arrive(tempty_bar(acc)); }
                    }
                    if constexpr (kPoolDirect) {
                        const bool wodd = (lane & 1) != 0, hodd = (lane & BW) != 0;
                        auto pool_store = [&](const int pair, const int mt, const uint32_t (&a)[32]) {
                            float m16[16], m8[8];
#pragma unroll
                            for (int k = 0; k < 16; ++k) {          // across w: the even lane keeps channels 0..15, the odd lane 16..31
                                const float lo = __uint_as_float(a[k]), hi = __uint_as_float(a[16 + k]);
                                const float recv = __shfl_xor_sync(0xffffffffu, wodd ? lo : hi, 1);
                                if constexpr (MASKSUM) m16[k] = (wodd ? hi : lo) + recv;
                                else m16[k] = fmaxf(wodd ? hi : lo, recv);
                            }
#pragma unroll
                            for (int k = 0; k < 8; ++k) {           // across h: the even row keeps the first 8 of those, the odd row the last 8
                                const float recv = __shfl_xor_sync(0xffffffffu, hodd ? m16[k] : m16[8 + k], BW);
                                if constexpr (MASKSUM) m8[k] = (hodd ? m16[8 + k] : m16[k]) + recv;
                                else m8[k] = fmaxf(hodd ? m16[8 + k] : m16[k], recv);
                            }
                            const int cs = (pair % kChunksPerTile) * CW + (wodd ? 16 : 0) + (hodd ? 8 : 0);
                            if constexpr (!MASKSUM) {
                                const float4 s0 = *reinterpret_cast<const float4*>(ss + cs), s1 = *reinterpret_cast<const float4*>(ss + cs + 4);
                                const float sh[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
                                for (int k = 0; k < 8; ++k) m8[k] = act_fn<ACT>(m8[k] + sh[k], p.act);   // max(a, b) + s == max(a + s, b + s)
                            }
                            size_t po = 0;
                            bool lv = false;
#pragma unroll
                            for (int m2 = 0; m2 < MT; ++m2)
                                if (m2 == mt) { po = pix_off[m2]; lv = live[m2]; }
                            if constexpr (MASKSUM) {   // a 2-term float sum is exact-commutative: every lane of a window forms the same sums
                                const uint4 rv = lv ? __ldg(reinterpret_cast<const uint4*>(p.ref + po + cbase + cs)) : make_uint4(0u, 0u, 0u, 0u);
                                const uint32_t rw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                                for (int k = 0; k < 8; ++k) {   // bf16 > 0: sign bit clear and not +0
                                    const uint32_t b = (rw[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
                                    m8[k] = (b != 0u && b < 0x8000u) ? m8[k] : 0.0f;
                                }
                            }
                            uint4 pk;
                            pk.x = pack_bf16x2(m8[0], m8[1]); pk.y = pack_bf16x2(m8[2], m8[3]);
                            pk.z = pack_bf16x2(m8[4], m8[5]); pk.w = pack_bf16x2(m8[6], m8[7]);
                            if (lv) __stcg(reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.out) + po + cbase + cs), pk);
                        };
                        pool_store(pa, mta < MT ? mta : 0, ra);
                        if (two) pool_store(pb, mtb < MT ? mtb : 0, rb);
                        GANREV_TRE(3, it * 4 + i0);
                        continue;
                    }
                    float va[32], vb[32];
                    math(pa, ra, va);
                    if (two && !kStoreEarly) math(pb, rb, vb);
                    GANREV_TRE(1, it * 4 + i0);
                    // tma_hybrid: the first chunk of a round leaves through the read-back / st.global path (its buffer is free at once),
                    // the second through a TMA store whose shared-memory read then has a whole round to complete -- no chunk waits
                    store(pa, mta < MT ? mta : 0, va, p.tma_store && !(p.tma_hybrid && two));
                    GANREV_TRE(2, it * 4 + i0);
                    if (two && kStoreEarly) math(pb, rb, vb);   // the first chunk's TMA store reads its staging buffer while the second chunk's math runs
                    if (two) store(pb, mtb < MT ? mtb : 0, vb, p.tma_store != 0);
                    GANREV_TRE(3, it * 4 + i0);
                }
            }
            if (!run) {
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) { if (CG == 2) mbar_arrive_cta(tempty_bar(acc), 0); else mbar_arrive(tempty_bar(acc)); }
            }
            if (etid == 0) GANREV_TR(5, it);
            }   // !FUSE3
        }
    }

    if (p.tma_store) tma_store_wait_read();                  // pending bulk stores have read their shared-memory source
    tcgen05_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();   // the leader's MMAs read the peer's smem: nobody leaves early
    if (warp == 2) {
        tcgen05_fence_after();
        if (CG == 2) tmem_dealloc_cg2<C::kTmemCols>(tmem_base); else tmem_dealloc<C::kTmemCols>(tmem_base);
    }
}

}  // namespace tc
}  // namespace ganrev

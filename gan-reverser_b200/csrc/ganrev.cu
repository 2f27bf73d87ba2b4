// ganrev.cu -- C ABI of libganrev_cuda.so (include/ganrev.h): context, weight preparation,
// chunked G / R pipelines, database ops, NCCL plumbing.  sm_100a only, no CPU fallback.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <memory>

#include "common.cuh"
#include "conv_simt.cuh"
#include "conv_tc.cuh"
#include "conv1_tc.cuh"
#include "layers.cuh"
#include "scan.cuh"
#include "search_tc.cuh"
#include "label_tc.cuh"
#include "stream_tc.cuh"
#include "nearest_tc.cuh"
#include "train.cuh"
#include "kmeans_tc.cuh"
#include "refine.cuh"

using namespace ganrev;

// =================================================================================
// context
// =================================================================================
constexpr int kMaxDevices = 64;   // per-device caches of kernel attributes

struct TcLayer {
    std::string name;
    ConvGemm g{};
    int NT = 0, MT = 1, NDY = 1, CG = 1, Ktot = 0;
    bool bres = false;
    size_t smem_bytes = 0;
    DevBuf w, shift;
    CUtensorMap tmB{};
    CUtensorMap tmO{};            // output map of the current launch (TMA-store layers)
    double flops_per_img = 0.0;   // executed MAC*2 per image (phase form counts the folded work)
    double bytes_per_img = 0.0;   // activation in + out per image
};

struct GModel {
    bool loaded = false;
    int C = 0, H = 0, W = 0, nd = 0, kpad = 0, F = 0;
    TcLayer lin, c1, c2, c3;   // c3 = pass 1 of the last conv (per-pixel tap products)
    DevBuf b3;
    DevBuf w3f;                // fp32 [9][128] tap-major weights of the last conv for the fused conv2 epilogue
    bool fuse3 = false;
    int cta_pairs = 0;         // ctx->cta_pairs at ganrev_load_G: the refinement's backward layers are built with it too
    std::vector<float> blob;   // host copy of the fp32 weight blob: the refinement's backward layers are built from it on first use
};
// Noise-vector refinement (ganrev_refine_l2): G's backward layers and the activations one chunk keeps for them.  Built on the
// first refine call, dropped when G is reloaded, so no other call's memory, launches or timings change.
struct GRefine {
    bool built = false;
    TcLayer c2t, c1t, lint;    // conv2^T, conv1^T (MASKSUM pooled epilogue), Linear^T (fp32 out)
    DevBuf w3t;                // fp32 [9][C][128] forward weights of the last conv for g_conv3_adjoint_kernel
    DevBuf h0, h1, h2, y, glin, m, v, zs, dist;   // per chunk: activations, G(z), W_lin^T(s0 e0), Adam moments; z / distances (debug call)
};
struct RModel {
    bool loaded = false;
    int C = 0, H = 0, W = 0, nd = 0, tanh_out = 0;
    DevBuf c1pack;              // CUDA-core conv1 (conv_impl 1): fp32 weights + scale + shift
    DevBuf c1w, c1shift;        // tcgen05 conv1: bf16 [64][KP] weights (BN scale folded, hi|lo halves), shift[64]
    TcLayer c2, c3, c4, c5, c6, l1, l2;
};

struct NcclApi {
    void* h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// R training state (train.cuh): fp32 parameters in weight-blob layout, Adam moments, step count, activations of one batch
struct TrainR {
    bool ready = false;
    int C = 0, H = 0, W = 0, nd = 0, tanh_out = 0, fixer = 0;
    size_t n_floats = 0;
    long long t = 0;
    DevBuf P, Gd, M, V, flags, work, masks, partial, lossbuf;
    size_t cw[6], cb[6], cg[6], cbe[6], crm[6], crv[6];   // blob offsets (floats) of conv i: weight, bias, BN gamma, beta, running mean, var
    size_t l1w, l1b, l1g, l1be, l1rm, l1rv, l2w, l2b;
    int ci[6], co[6];
    int B_cap = 0;
};

struct ganrev_ctx {
    int device = 0, num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;   // host <-> device copies of forward_G / forward_R run chunk by chunk beside the kernels (created on first use)
    std::vector<cudaEvent_t> io_events;
    bool copies_pending = false;
    std::string err;
    int64_t chunk = 0;            // images per pipeline chunk; 0 = auto (8192 32x32 faces' worth of pixels, see chunk_for)
    int conv_impl = 0;
    int tma_hybrid = 0;           // see ConvGemm::tma_hybrid (A/B)
    int ups_cycles = 512;         // a pipeline stage carries enough units for this many MMA cycles (one mbarrier round trip per stage); read at load time
    int pdl = 0;                  // conv layers launched with programmatic stream serialization (prologue overlaps the previous kernel's tail);
                                  // measured +0.4 % on the resident G->R chain (tools/ab_total.py pdl 0 1: within noise), so off by default
    int xpose2 = 1;               // double store-transpose buffers in the TMA-store epilogue (see build_tc_layer); 0 = single (A/B)
    int fuse_conv3 = 1;           // the last conv's tap products are computed in G conv2's epilogue: 1 = when C == 1 (free there: the epilogue has the
                                  // slack), 2 = also C == 3 (measured: 27 taps make conv2 epilogue-bound, 8.3 -> 15.3 ms per 4096 64x64 faces), 0 = never
    int tma_store = 1;            // TMA bulk tensor stores in the conv epilogue where the layer allows (0 = st.global everywhere; A/B)
    int search_tc = 1;            // tensor-core candidate filter + exact re-score for many-query searches (0 = fmaf-chain kernels only; A/B)
    uint64_t tc_searches = 0, tc_fallbacks = 0;   // searches served by the tensor-core path / re-run on the fmaf-chain kernels
    int label_tc = 0;             // 1 = tensor-core labelling for k <= 32, d <= 128 (label_tc.cuh; bit-exact, measured no faster than rtile_kernel yet: off)
    int stream_tc = 1;            // TMA -> tf32 tcgen05 filter pipeline for <= 32 needles / centroids (stream_tc.cuh; 0 = the fmaf-chain streaming kernels; A/B)
    int kmeans_tc = 1;            // tensor-core labelling for 32 < k (kmeans_tc.cuh): approximate scores, exact chains only for near-ties
    int rtile = 1;                // register-tiled kmeans / cosine-min kernels for 9 <= k <= 32 (0 = the one-thread-per-row streaming kernels; A/B)
    int cta_pairs = 0x1f;     // which layers use tcgen05 cta_group::2 CTA pairs (bit0 G conv1, bit1 G conv2, bit2 R conv2/3,
                              // bit3 R conv4, bit4 R conv5/6); takes effect at the next ganrev_load_*.  Default = measured best.
    int dbg = 0;
    DevBuf trace;
    std::string trace_layer;
    uint64_t launches = 0;
    int* d_err_flag = nullptr;
    EncodeTiledFn encode = nullptr;
    // profiling
    bool prof_on = false;
    std::vector<ProfEntry> prof;
    std::map<std::string, int> prof_idx;
    std::vector<ProfPending> pending;
    std::vector<cudaEvent_t> ev_pool;
    // models
    GModel G;
    GRefine GR;
    RModel R[2];
    // resident buffers + activation arena
    DevBuf buf[GANREV_BUF_COUNT];
    int64_t buf_rows[GANREV_BUF_COUNT] = {0, 0, 0, 0, 0, 0};
    int gC = 0, gH = 0, gW = 0, gnd = 0;   // the one geometry every loaded model and resident buffer shares (0 = none yet)
    DevBuf arena[2], noise_bf16, stage_a, stage_b, l2buf, thr, flags;
    int64_t l2_valid = 0;                  // entries of l2buf written by the last fix_l2 / l2 / anomaly_flags call
    DevBuf nn_partial, nn_ids, nn_dist, nn_flag, nn_all;   // ganrev_nearest_l2 scratch
    DevBuf amb, pdb, pq, tc_thr, tc_cnt, tc_cand, tc_pairs, tc_keys, tc_special, tc_flags, tc_dump;   // search_tc.cuh: packed split-bf16 operands, candidates
    bool pdb_valid = false;                // pdb / tc_special describe the current database
    DevBuf tfs_aux;                        // stream_tc.cuh: published k-th scores [32 u32] | stats [4 u64]
    uint64_t tfs_launches = 0;
    DevBuf qsel, shard;                    // radix-select state + histogram; row-shard bookkeeping (world + 2 int64)
    // database
    DevBuf db, rdb, maxabs;
    const float* db_ptr = nullptr;         // rows of the database: db.p (own copy) or the resident ATTRS0 buffer (alias)
    bool db_alias = false;
    int64_t db_n = 0, db_offset = 0, db_total = 0;
    int db_d = 0;
    float db_maxabs = 0.0f;
    DevBuf q, rq, c2, partial, keys, keys_all, ids, scores;
    DevBuf cen, acc, cnt, total, labels, cosv, tcounts, mids, mcnt, mmean;
    bool assigned = false;
    int assigned_k = 0;
    TrainR train;
    // nccl
    NcclApi nccl;
    ncclComm_t comm = nullptr;
    int world = 1, rank = 0;
};

static int fail(ganrev_ctx* c, int code, const char* fmt, ...) {
    char tmp[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tmp, sizeof(tmp), fmt, ap);
    va_end(ap);
    if (c) c->err = tmp;
    return code;
}
#define CU_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess) return fail(ctx, GANREV_ECUDA, "%s failed: %s (%s:%d)", #expr,     \
                                           cudaGetErrorString(e_), __FILE__, __LINE__);           \
    } while (0)
#define RC_TRY(expr)            \
    do {                        \
        int rc_ = (expr);       \
        if (rc_ != GANREV_OK) return rc_; \
    } while (0)

static int ensure(ganrev_ctx* ctx, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap && b.p) return GANREV_OK;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    if (bytes == 0) bytes = 256;
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) return fail(ctx, GANREV_ENOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    b.cap = bytes;
    return GANREV_OK;
}
static void release(DevBuf& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
}

// ---- profiling helpers -------------------------------------------------------------
struct ProfScope {
    ganrev_ctx* ctx;
    ProfPending pp{};
    bool on;
    // count = false: a library (NCCL) call, timed but not one of OUR kernel launches
    ProfScope(ganrev_ctx* c, const std::string& name, double flops, double bytes, bool count = true) : ctx(c), on(c->prof_on) {
        if (count) ctx->launches++;
        if (!on) return;
        auto it = ctx->prof_idx.find(name);
        int idx;
        if (it == ctx->prof_idx.end()) {
            idx = static_cast<int>(ctx->prof.size());
            ProfEntry e; e.name = name;
            ctx->prof.push_back(e);
            ctx->prof_idx[name] = idx;
        } else idx = it->second;
        ctx->prof[idx].launches++;
        ctx->prof[idx].flops += flops;
        ctx->prof[idx].bytes += bytes;
        pp.entry = idx;
        pp.e0 = take(); pp.e1 = take();
        cudaEventRecord(pp.e0, ctx->stream);
    }
    cudaEvent_t take() {
        if (!ctx->ev_pool.empty()) { cudaEvent_t e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(pp.e1, ctx->stream);
        ctx->pending.push_back(pp);
    }
};
static void prof_resolve(ganrev_ctx* ctx) {
    for (auto& pp : ctx->pending) {
        float ms = 0.0f;
        if (cudaEventSynchronize(pp.e1) == cudaSuccess && cudaEventElapsedTime(&ms, pp.e0, pp.e1) == cudaSuccess)
            ctx->prof[pp.entry].total_ms += ms;
        ctx->ev_pool.push_back(pp.e0);
        ctx->ev_pool.push_back(pp.e1);
    }
    ctx->pending.clear();
}

static int finish(ganrev_ctx* ctx) {
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (ctx->copies_pending) {
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->copy_in);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->copy_out);
        ctx->copies_pending = false;
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        int flag = 0;
        return fail(ctx, GANREV_ECUDA, "device error: %s (pipeline watchdog flag unreadable=%d)", cudaGetErrorString(e), flag);
    }
    int flag = 0;
    cudaMemcpy(&flag, ctx->d_err_flag, sizeof(int), cudaMemcpyDeviceToHost);
    if (flag != 0) return fail(ctx, GANREV_ECUDA, "tcgen05 pipeline watchdog fired (code %d)", flag);
    return GANREV_OK;
}

// =================================================================================
// host-side weight preparation
// =================================================================================
static inline uint16_t f2bf(float f) {   // round-to-nearest-even, NaN preserved
    uint32_t u; memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40u);
    const uint32_t r = 0x7fffu + ((u >> 16) & 1u);
    return static_cast<uint16_t>((u + r) >> 16);
}
struct BnFold {
    std::vector<float> scale, shift;
};
// eval-mode BatchNorm after a layer with bias b:  y = (x + b - mean) * g/sqrt(var+eps) + beta
static BnFold fold_bn(const float* bias, const float* g, const float* beta, const float* mean, const float* var, int n, int pad) {
    BnFold f;
    f.scale.assign(pad, 0.0f); f.shift.assign(pad, 0.0f);
    for (int i = 0; i < n; ++i) {
        const float s = g[i] / std::sqrt(var[i] + 1e-5f);
        f.scale[i] = s;
        f.shift[i] = beta[i] + (bias[i] - mean[i]) * s;
    }
    return f;
}
static int upload(ganrev_ctx* ctx, DevBuf& b, const void* src, size_t bytes) {
    RC_TRY(ensure(ctx, b, bytes));
    CU_TRY(cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice));
    return GANREV_OK;
}
static int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }
static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

enum LayerKind { KIND_LINEAR = 0, KIND_CONV3 = 1, KIND_UPCONV3 = 2 };

static int make_tmB(ganrev_ctx* ctx, TcLayer& L) {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(L.Ktot), static_cast<cuuint64_t>(L.g.nphase) * L.g.cout_pad};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(L.Ktot) * 2};
    const cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(L.NT / L.CG)};
    const cuuint32_t es[2] = {1u, 1u};
    CUresult r = ctx->encode(&L.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, L.w.p, dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, GANREV_ECUDA, "cuTensorMapEncodeTiled(B, %s) failed: %d", L.name.c_str(), (int)r);
    return GANREV_OK;
}

struct LayerDef {
    const char* name;
    LayerKind kind;
    int NT, MT;              // N tile, accumulators per CTA
    int cg;                  // 1, or 2 = CTA pairs (tcgen05 cta_group::2: M = 256 per MMA, each CTA holds half of B)
    bool want_bres;          // keep the whole weight matrix resident in smem when it fits
    int Hin, Win, Cin;
    int cout_real, n_tiles;
    int Hout, Wout, out_cstride;
    int pool, act;
    float post_scale;
    int out_fp32;
    bool nchw;
};

// w: conv weights [cout_real][Cin][3][3] (KIND_CONV3 / KIND_UPCONV3) or a ready matrix
// [n_tiles*NT][Cin] (KIND_LINEAR).  BatchNorm arrives folded in `bn` (cout_pad entries).
static int build_tc_layer(ganrev_ctx* ctx, TcLayer& L, const LayerDef& d, const float* w, const BnFold& bn) {
    L.name = d.name;
    L.NT = d.NT;
    L.CG = d.cg;
    ConvGemm& g = L.g;
    g = ConvGemm{};
    g.Hin = d.Hin; g.Win = d.Win; g.Cin = d.Cin;
    if (d.Cin % 64 != 0) return fail(ctx, GANREV_EINVAL, "layer %s: Cin=%d not a multiple of 64", d.name, d.Cin);
    g.cin_chunks = d.Cin / 64;
    g.n_tiles = d.n_tiles; g.cout_pad = d.n_tiles * d.NT; g.cout_real = d.cout_real;
    if (d.nchw) { g.out_sN = static_cast<long long>(d.out_cstride) * d.Hout * d.Wout; g.out_sP = 1; g.out_sC = d.Hout * d.Wout; }
    else        { g.out_sN = static_cast<long long>(d.out_cstride) * d.Hout * d.Wout; g.out_sP = d.out_cstride; g.out_sC = 1; }
    g.Hout = d.Hout; g.Wout = d.Wout; g.up = d.kind == KIND_UPCONV3 ? 2 : 1; g.pool = d.pool; g.act = d.act;
    if (d.post_scale != 1.0f) return fail(ctx, GANREV_EINVAL, "layer %s: fold the post-scale into the next layer's weights", d.name);
    g.post_scale = d.post_scale; g.out_fp32 = d.out_fp32;
    g.err_flag = ctx->d_err_flag;

    // ---- M tile and tap groups.  Halo reuse needs a whole 128-pixel tile inside one image.
    const bool halo = d.kind != KIND_LINEAR && d.Hin * d.Win >= 128 && d.Win >= 8;
    int BW, BH, BN;
    if (halo) { BW = std::min(d.Win, 16); BH = 128 / BW; BN = 1; }
    else      { BW = std::min(d.Win, d.pool ? 16 : 128); BH = std::min(d.Hin, 128 / BW); BN = 128 / (BW * BH); }
    g.lgBW = ilog2(BW); g.lgBH = ilog2(BH); g.lgBN = ilog2(BN);
    g.tiles_w = d.Win / BW; g.tiles_h = d.Hin / BH;
    g.lgTW = ilog2(g.tiles_w); g.lgTH = ilog2(g.tiles_h);
    g.lgNT = is_pow2(g.n_tiles) ? ilog2(g.n_tiles) : -1;
    g.nphase = d.kind == KIND_UPCONV3 ? 4 : 1;
    if (d.kind == KIND_LINEAR) { g.ngroups = 1; g.ndy = 1; }
    else if (d.kind == KIND_CONV3) {
        if (halo) { g.ngroups = 3; g.ndy = 3; for (int x = 0; x < 3; ++x) { g.gdx[0][x] = static_cast<int8_t>(x - 1); g.gdy0[0][x] = -1; } }
        else      { g.ngroups = 9; g.ndy = 1; for (int t = 0; t < 9; ++t) { g.gdy0[0][t] = static_cast<int8_t>(t / 3 - 1); g.gdx[0][t] = static_cast<int8_t>(t % 3 - 1); } }
    } else {   // phase p = a*2 + b reads low-res rows a-1..a and columns b-1..b
        for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 2; ++b) {
                const int ph = a * 2 + b;
                if (halo) { g.ngroups = 2; g.ndy = 2; for (int x = 0; x < 2; ++x) { g.gdx[ph][x] = static_cast<int8_t>(b - 1 + x); g.gdy0[ph][x] = static_cast<int8_t>(a - 1); } }
                else      { g.ngroups = 4; g.ndy = 1; for (int t = 0; t < 4; ++t) { g.gdy0[ph][t] = static_cast<int8_t>(a - 1 + t / 2); g.gdx[ph][t] = static_cast<int8_t>(b - 1 + t % 2); } }
            }
    }
    L.NDY = g.ndy;
    L.MT = d.MT;
    if (!halo && !(d.kind == KIND_UPCONV3 && d.NT == 256)) L.CG = 1;   // CTA-pair variants exist for the halo layers and G conv1
    g.units = g.ngroups * g.cin_chunks;
    const int ntap = g.ngroups * g.ndy;
    L.Ktot = ntap * d.Cin;

    // ---- weight matrix [nphase*cout_pad][Ktot], K = (g*ndy + j)*Cin + ci.  The folded BatchNorm scale is
    // multiplied into each output row BEFORE the one rounding to bf16, so the epilogue only adds `shift`.
    std::vector<uint16_t> wb(static_cast<size_t>(g.nphase) * g.cout_pad * L.Ktot, 0);
    if (d.kind == KIND_LINEAR) {
        for (int co = 0; co < g.cout_pad; ++co)
            for (int ci = 0; ci < d.Cin; ++ci) wb[static_cast<size_t>(co) * d.Cin + ci] = f2bf(w[static_cast<size_t>(co) * d.Cin + ci] * bn.scale[co]);
    } else {
        // nearest-upsample x2 then 3x3/pad1 == four 2x2 convolutions on the low-res input: output row
        // 2y+a reads low-res rows {y-1: ky=0 | y: ky=1,2} (a=0) or {y: ky=0,1 | y+1: ky=2} (a=1).
        static const int S[2][2][2] = {{{0, 0}, {1, 2}}, {{0, 1}, {2, 2}}};   // S[a][t] = {first, last} ky
        for (int ph = 0; ph < g.nphase; ++ph)
            for (int gi = 0; gi < g.ngroups; ++gi)
                for (int j = 0; j < g.ndy; ++j) {
                    const int dy = g.gdy0[ph][gi] + j, dx = g.gdx[ph][gi];
                    int ky0, ky1, kx0, kx1;
                    if (d.kind == KIND_CONV3) { ky0 = ky1 = dy + 1; kx0 = kx1 = dx + 1; }
                    else {
                        const int a = ph >> 1, b = ph & 1, ty = dy - (a - 1), tx = dx - (b - 1);
                        ky0 = S[a][ty][0]; ky1 = S[a][ty][1]; kx0 = S[b][tx][0]; kx1 = S[b][tx][1];
                    }
                    for (int co = 0; co < d.cout_real; ++co)
                        for (int ci = 0; ci < d.Cin; ++ci) {
                            double sum = 0.0;
                            for (int ky = ky0; ky <= ky1; ++ky)
                                for (int kx = kx0; kx <= kx1; ++kx) sum += w[((static_cast<size_t>(co) * d.Cin + ci) * 3 + ky) * 3 + kx];
                            wb[(static_cast<size_t>(ph) * g.cout_pad + co) * L.Ktot + static_cast<size_t>(gi * g.ndy + j) * d.Cin + ci] = f2bf(static_cast<float>(sum * bn.scale[co]));
                        }
                }
    }
    RC_TRY(upload(ctx, L.w, wb.data(), wb.size() * 2));
    RC_TRY(upload(ctx, L.shift, bn.shift.data(), bn.shift.size() * 4));
    g.B = reinterpret_cast<const bf16*>(L.w.p);
    g.shift = reinterpret_cast<const float*>(L.shift.p);
    RC_TRY(make_tmB(ctx, L));

    // ---- shared-memory plan: [resident weights][stages x (ups units)][barriers, shift]
    g.a_unit_bytes = (BH + g.ndy - 1) * BW * BN * 128;
    g.b_kb_bytes = (d.NT / L.CG) * 128;          // this CTA's share of a 64-wide weight tile
    g.dy_stride_bytes = BW * BN * 128;
    // barriers, shift (double-buffered), store-transpose buffers (xp per epilogue warp)
    const size_t wbytes = static_cast<size_t>(g.units) * g.ndy * g.b_kb_bytes;
    auto plan = [&](int xp) -> bool {
        const int tail = ((2 * tc::kMaxStages + 5) * 8 + 24 + 2 * d.NT * 4 + 1023) / 1024 * 1024 + xp * tc::kEpiWarps * 32 * 64;
        const int budget = tc::kSmemBudget - 1024 - tail;
        L.bres = d.want_bres && g.nphase == 1 && g.n_tiles == 1 && wbytes + 2 * static_cast<size_t>(L.MT) * g.a_unit_bytes <= static_cast<size_t>(budget);
        for (;;) {
            const int res = L.bres ? static_cast<int>(wbytes) : 0;
            g.unit_bytes = L.MT * g.a_unit_bytes + (L.bres ? 0 : g.ndy * g.b_kb_bytes);
            const int cyc_unit = L.MT * g.ndy * 4 * std::max(d.NT / 2, 32);          // MMA cycles per unit
            // units per stage: one mbarrier round trip per >= ups_cycles MMA cycles.  G's Up+Conv 512->256 (N = 256: 548 MMA cycles per unit,
            // 32 units per item) measured 5 % faster with two units per stage (same-box A/B against conv2, tools/ab_option.py ups_cycles
            // 512 1024); the Linear layers measured 2 % slower with it, the others do not change
            const int tgt = (d.kind == KIND_UPCONV3 && d.NT == 256) ? std::max(ctx->ups_cycles, 1024) : ctx->ups_cycles;
            g.ups = std::max(1, std::min({4, g.units, (tgt + cyc_unit - 1) / cyc_unit}));
            while (g.ups > 1 && (budget - res) / (g.ups * g.unit_bytes) < 3) --g.ups;
            g.stage_bytes = g.ups * g.unit_bytes;
            g.stages = std::min(tc::kMaxStages, (budget - res) / g.stage_bytes);
            if (g.stages >= 2) { L.smem_bytes = static_cast<size_t>(res) + static_cast<size_t>(g.stages) * g.stage_bytes + tail + 1024; g.xpose2 = xp == 2; return true; }
            if (L.bres) { L.bres = false; continue; }
            return false;
        }
    };
    // Two store-transpose buffers per epilogue warp let a TMA store's shared-memory read overlap the next chunk's math (with one
    // buffer every chunk waits for the previous store).  Measured per layer (tools/ab_option.py xpose2 0 1 2, 32768 faces): G's Linear
    // (K = 128, store-bound) 2.33 -> 2.00 ms; R conv2 +5 % and R Linear1 +13 % (the 16 KB cost them a pipeline stage), R conv4 / conv5
    // unchanged.  xpose2 = 1 (default): G's Linear only; 2: every plain bf16 layer (A/B); 0: nowhere.
    const bool plain = !d.pool && !d.out_fp32 && d.kind != KIND_UPCONV3 && !d.nchw && d.cout_real == g.cout_pad && d.NT % 32 == 0;
    const bool want2 = plain && (ctx->xpose2 == 2 || (ctx->xpose2 == 1 && !strcmp(d.name, "g_linear")));
    if (!(want2 && plan(2)) && !plan(1)) return fail(ctx, GANREV_EINVAL, "layer %s does not fit in shared memory", d.name);
    const double px_in = static_cast<double>(d.Hin) * d.Win;
    L.flops_per_img = 2.0 * px_in * g.nphase * (d.out_fp32 ? d.cout_real : g.cout_pad) * L.Ktot;   // zero-padded output lanes are not work
    L.bytes_per_img = 2.0 * px_in * d.Cin + (d.out_fp32 ? 4.0 : 2.0) * d.Hout * d.Wout * d.cout_real;
    return GANREV_OK;
}

static int check_geom(ganrev_ctx* ctx, int C, int H, int W, int nd) {
    if (!(C == 1 || C == 3)) return fail(ctx, GANREV_EINVAL, "C must be 1 or 3 (got %d)", C);
    if (!is_pow2(H) || !is_pow2(W) || H < 16 || W < 16 || H > 256 || W > 256)
        return fail(ctx, GANREV_EINVAL, "H, W must be powers of two in [16,256] (got %dx%d)", H, W);
    if (nd < 1 || nd > 4096) return fail(ctx, GANREV_EINVAL, "noise_dim out of range: %d", nd);
    return GANREV_OK;
}

// =================================================================================
// layer launches
// =================================================================================
template <int NT, int MT, int NDY, bool BRES, int ACT, bool POOL, bool OUT_FP32, int CG, int FUSE3 = 0, bool MASKSUM = false>
static int launch_tc(ganrev_ctx* ctx, const TcLayer& L, const CUtensorMap& tmA, const ConvGemm& g, int n_items) {
    auto kern = tc::conv_tc_kernel<NT, MT, NDY, BRES, ACT, POOL, OUT_FP32, CG, FUSE3, MASKSUM>;
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (L.smem_bytes > attr_max) {
        CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(L.smem_bytes)));
        attr_max = L.smem_bytes;
    }
    int grid = std::min(n_items * CG, ctx->num_sms);
    grid -= grid % CG;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(tc::kThreads);
    cfg.dynamicSmemBytes = L.smem_bytes;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (CG == 2) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = CG; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        ++na;
    }
    if (ctx->pdl) {   // programmatic dependent launch: this kernel's prologue may overlap the previous kernel's tail (conv_tc.cuh)
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    CU_TRY(cudaLaunchKernelEx(&cfg, kern, tmA, L.tmB, L.tmO, g, n_items));
    return GANREV_OK;
}
// The layer shapes of G3 / R_default map onto this fixed set of kernel variants
// (NT, MT, NDY, BRES, ACT, POOL, FP32OUT).  NDY=1 rows serve geometries too small for halo reuse.
static int dispatch_tc(ganrev_ctx* ctx, const TcLayer& L, const CUtensorMap& tmA, const ConvGemm& g, int n_items) {
#define TC_CASE_CG(NT_, MT_, NDY_, BRES_, ACT_, POOL_, FP32_, CG_)                                                      \
    if (L.NT == NT_ && L.MT == MT_ && L.NDY == NDY_ && L.bres == BRES_ && (ACT_ == tc::ACT_RUNTIME || g.act == ACT_) && \
        (g.pool != 0) == POOL_ && (g.out_fp32 != 0) == FP32_ && L.CG == CG_)                                            \
        return launch_tc<NT_, MT_, NDY_, BRES_, ACT_, POOL_, FP32_, CG_>(ctx, L, tmA, g, n_items);
#define TC_CASE(NT_, MT_, NDY_, BRES_, ACT_, POOL_, FP32_) TC_CASE_CG(NT_, MT_, NDY_, BRES_, ACT_, POOL_, FP32_, 1)
    if (g.w3 != nullptr) {   // G Up+Conv 256->128 with the last conv's tap products fused into the epilogue
#define TC_FUSED(NDY_, CG_, C_) \
        if (L.NT == 128 && L.MT == 2 && L.NDY == NDY_ && L.CG == CG_ && g.w3_c == C_) return launch_tc<128, 2, NDY_, false, ACT_RELU, false, false, CG_, C_>(ctx, L, tmA, g, n_items);
        TC_FUSED(2, 2, 1) TC_FUSED(2, 1, 1) TC_FUSED(1, 1, 1)
        TC_FUSED(2, 2, 3) TC_FUSED(2, 1, 3) TC_FUSED(1, 1, 3)
#undef TC_FUSED
        return fail(ctx, GANREV_EINVAL, "no fused tap-product variant for layer %s", L.name.c_str());
    }
    if (g.ref != nullptr) {  // G's backward convs (refinement): 2x2 sum-pool * [forward activation > 0]
#define TC_MASKSUM(NDY_, CG_) \
        if (L.NT == 128 && L.MT == 2 && L.NDY == NDY_ && !L.bres && g.pool && !g.out_fp32 && L.CG == CG_) return launch_tc<128, 2, NDY_, false, ACT_NONE, true, false, CG_, 0, true>(ctx, L, tmA, g, n_items);
        TC_MASKSUM(3, 2) TC_MASKSUM(3, 1) TC_MASKSUM(1, 1)
#undef TC_MASKSUM
        return fail(ctx, GANREV_EINVAL, "no sum-pool / mask variant for layer %s", L.name.c_str());
    }
    // CTA-pair (cta_group::2) variants of the halo layers
    TC_CASE_CG(256, 1, 1, false, ACT_RELU, false, false, 2)   // G Up+Conv 512->256
    TC_CASE_CG(256, 1, 2, false, ACT_RELU, false, false, 2)
    TC_CASE_CG(128, 2, 2, false, ACT_RELU, false, false, 2)   // G Up+Conv 256->128
    TC_CASE_CG(64, 2, 3, true, ACT_ELU, false, false, 2)      // R Conv 64->64
    TC_CASE_CG(64, 2, 3, true, ACT_ELU, true, false, 2)
    TC_CASE_CG(64, 4, 3, true, ACT_ELU, false, false, 2)      // ... four sub-tiles per item (8 x 64 = 512 TMEM columns, double-buffered)
    TC_CASE_CG(64, 4, 3, true, ACT_ELU, true, false, 2)
    TC_CASE_CG(128, 1, 3, true, ACT_ELU, false, false, 2)     // R Conv 64->128
    TC_CASE_CG(128, 2, 3, true, ACT_ELU, false, false, 2)
    TC_CASE_CG(128, 2, 3, false, ACT_ELU, false, false, 2)    // R Conv 128->128
    TC_CASE_CG(128, 2, 3, false, ACT_ELU, true, false, 2)
    // G
    TC_CASE(256, 1, 1, false, ACT_RELU, false, false)      // Linear
    TC_CASE(256, 2, 1, false, ACT_RELU, false, false)      // Up+Conv 512->256 on < 128-pixel inputs
    TC_CASE(256, 2, 2, false, ACT_RELU, false, false)      // ... with halo reuse
    TC_CASE(128, 2, 1, false, ACT_RELU, false, false)      // Up+Conv 256->128
    TC_CASE(128, 2, 2, false, ACT_RELU, false, false)
    TC_CASE(16, 1, 1, false, ACT_NONE, false, true)        // last conv pass 1: per-pixel tap products, C = 1
    TC_CASE(32, 1, 1, false, ACT_NONE, false, true)        // ... C = 3
    // R
    TC_CASE(64, 2, 3, true, ACT_ELU, false, false)         // Conv 64->64
    TC_CASE(64, 2, 3, true, ACT_ELU, true, false)          // Conv 64->64 + MaxPool
    TC_CASE(128, 1, 3, true, ACT_ELU, false, false)        // Conv 64->128
    TC_CASE(128, 1, 1, true, ACT_ELU, false, false)
    TC_CASE(128, 2, 3, false, ACT_ELU, false, false)       // Conv 128->128
    TC_CASE(128, 2, 3, false, ACT_ELU, true, false)        // Conv 128->128 + x0.75 + MaxPool
    TC_CASE(128, 2, 1, false, ACT_ELU, false, false)
    TC_CASE(128, 2, 1, false, ACT_ELU, true, false)
    TC_CASE(64, 1, 1, false, ACT_ELU, false, false)
    TC_CASE(256, 1, 1, false, ACT_ELU, false, false)       // Linear 8192->512
    TC_CASE(32, 1, 1, false, tc::ACT_RUNTIME, false, true) // Linear 512->nd (+Tanh)
    TC_CASE(64, 1, 1, false, tc::ACT_RUNTIME, false, true)
    TC_CASE(128, 1, 1, false, tc::ACT_RUNTIME, false, true)
    TC_CASE(256, 1, 1, false, tc::ACT_RUNTIME, false, true)
#undef TC_CASE
#undef TC_CASE_CG
    return fail(ctx, GANREV_EINVAL, "no tcgen05 kernel variant for layer %s (NT=%d MT=%d NDY=%d bres=%d act=%d pool=%d fp32=%d cg=%d)", L.name.c_str(),
                L.NT, L.MT, L.NDY, (int)L.bres, g.act, g.pool, g.out_fp32, L.CG);
}

static int run_layer(ganrev_ctx* ctx, TcLayer& L, const void* in, void* out, int n_img, int64_t n_cap) {
    ConvGemm g = L.g;
    g.A = reinterpret_cast<const bf16*>(in);
    g.out = out;
    g.n_img = n_img;
    g.dbg = ctx->dbg;
    g.trace = (ctx->trace.p && L.name == ctx->trace_layer) ? static_cast<long long*>(ctx->trace.p) : nullptr;
    const int BN = 1 << g.lgBN;
    const int tiles_n = (n_img + BN - 1) / BN;
    g.total_tiles = tiles_n * g.tiles_h * g.tiles_w;
    const int mgroups = (g.total_tiles + L.MT * L.CG - 1) / (L.MT * L.CG);
    const int n_items = mgroups * g.nphase * g.n_tiles;
    const double px_out = static_cast<double>(g.Hout) * g.Wout;
    // fused tap products: + 9*C x 128 MACs per output pixel on the FMA pipe, 36*C B of planes instead of the 256 B bf16 activation
    const double fl_img = L.flops_per_img + (g.w3 ? 2.0 * 9 * g.w3_c * 128 * px_out : 0.0), by_img = g.w3 ? L.bytes_per_img - 2.0 * 128 * px_out + 36.0 * g.w3_c * px_out : L.bytes_per_img;
    ProfScope ps(ctx, L.name, fl_img * n_img, by_img * n_img);
    if (ctx->conv_impl == 1) {
        const long long total = static_cast<long long>(n_img) * g.Hout * g.Wout * g.cout_real;
        conv_simt_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, ctx->stream>>>(g, total);
        CU_TRY(cudaGetLastError());
        return GANREV_OK;
    }
    CUtensorMap tmA;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(g.Cin), static_cast<cuuint64_t>(g.Win), static_cast<cuuint64_t>(g.Hin),
                                static_cast<cuuint64_t>(n_cap)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(g.Cin) * 2, static_cast<cuuint64_t>(g.Win) * g.Cin * 2,
                                   static_cast<cuuint64_t>(g.Hin) * g.Win * g.Cin * 2};
    const cuuint32_t box[4] = {64u, 1u << g.lgBW, (1u << g.lgBH) + static_cast<cuuint32_t>(g.ndy - 1), 1u << g.lgBN};
    const cuuint32_t es[4] = {1u, 1u, 1u, 1u};
    CUresult r = ctx->encode(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(in), dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, GANREV_ECUDA, "cuTensorMapEncodeTiled(A, %s) failed: %d", L.name.c_str(), (int)r);
    // Output map for the TMA-store epilogue: plain (no pool / upsample) bf16 NHWC layers with whole 32-channel chunks.  A lane
    // quarter's 32 pixels are one box {32 ch, bw, bh, bn} of the [n][Hout][Wout][channels] tensor; rows past n_img are clipped.
    // (pooled layers can use it too -- the epilogue packs the writer lanes densely -- but measured 1.5-4 % slower there: option value 2)
    g.tma_store = (ctx->tma_store && (!g.pool || ctx->tma_store == 2) && !g.out_fp32 && g.up == 1 && g.out_sC == 1 && g.cout_real == g.cout_pad && L.NT % 32 == 0) ? 1 : 0;
    g.tma_hybrid = (g.tma_store && !g.xpose2 && !g.pool) ? ctx->tma_hybrid : 0;
    L.tmO = tmA;
    {
        const int BW = 1 << g.lgBW, BH = 1 << g.lgBH;
        if (g.pool && (std::min(BW, 32) < 2 || std::min(BH, 32 / std::min(BW, 32)) < 2)) g.tma_store = 0;   // a lane quarter must hold whole 2x2 windows
    }
    if (g.tma_store) {
        const int BW = 1 << g.lgBW, BH = 1 << g.lgBH;
        int bw = std::min(BW, 32), bh = std::min(BH, 32 / bw);
        const int bn = 32 / (bw * bh);
        if (g.pool) { bw /= 2; bh /= 2; }                      // the pooled quarter: (bw/2) x (bh/2) pixels, packed densely by the epilogue
        const cuuint64_t odims[4] = {static_cast<cuuint64_t>(g.out_sP), static_cast<cuuint64_t>(g.Wout), static_cast<cuuint64_t>(g.Hout), static_cast<cuuint64_t>(n_img)};
        const cuuint64_t ostr[3] = {static_cast<cuuint64_t>(g.out_sP) * 2, static_cast<cuuint64_t>(g.Wout) * g.out_sP * 2, static_cast<cuuint64_t>(g.out_sN) * 2};
        const cuuint32_t obox[4] = {32u, static_cast<cuuint32_t>(bw), static_cast<cuuint32_t>(bh), static_cast<cuuint32_t>(bn)};
        r = ctx->encode(&L.tmO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, out, odims, ostr, obox, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(ctx, GANREV_ECUDA, "cuTensorMapEncodeTiled(out, %s) failed: %d", L.name.c_str(), (int)r);
    }
    return dispatch_tc(ctx, L, tmA, g, n_items);
}

// =================================================================================
// model loading
// =================================================================================
static void release_layer(TcLayer& L) { release(L.w); release(L.shift); }
static void release_refine(GRefine& R) {
    for (TcLayer* L : {&R.c2t, &R.c1t, &R.lint}) release_layer(*L);
    for (DevBuf* b : {&R.w3t, &R.h0, &R.h1, &R.h2, &R.y, &R.glin, &R.m, &R.v, &R.zs, &R.dist}) release(*b);
    R.built = false;
}

// One geometry per context: G, R and R_fixer of apply_r.lua share {C, H, W, noiseDim} (apply_r.lua:65-79), and the resident
// buffers are sized by it.  Loading a model of a DIFFERENT geometry therefore unloads the models of the old one and empties
// every resident buffer (and a database aliasing ATTRS0) -- nothing sized for the old geometry can be read or written afterwards.
static void adopt_geometry(ganrev_ctx* ctx, int C, int H, int W, int nd) {
    if (ctx->gC == C && ctx->gH == H && ctx->gW == W && ctx->gnd == nd) return;
    ctx->G.loaded = false;
    ctx->R[0].loaded = ctx->R[1].loaded = false;
    for (int b = 0; b < GANREV_BUF_COUNT; ++b) ctx->buf_rows[b] = 0;
    if (ctx->db_alias) { ctx->db_ptr = nullptr; ctx->db_alias = false; ctx->db_n = 0; ctx->assigned = false; }
    ctx->l2_valid = 0;
    ctx->gC = C; ctx->gH = H; ctx->gW = W; ctx->gnd = nd;
}

static int load_G_impl(ganrev_ctx* ctx, int C, int H, int W, int nd, const float* blob, size_t n_floats) {
    RC_TRY(check_geom(ctx, C, H, W, nd));
    const int sH = H / 4, sW = W / 4, HW0 = sH * sW, F = 512 * HW0;
    const size_t need = static_cast<size_t>(F) * nd + 5 * static_cast<size_t>(F) + 256u * 512 * 9 + 5 * 256 + 128u * 256 * 9 + 5 * 128 +
                        static_cast<size_t>(C) * 128 * 9 + C;
    if (n_floats != need) return fail(ctx, GANREV_EINVAL, "G blob has %zu floats, expected %zu", n_floats, need);
    adopt_geometry(ctx, C, H, W, nd);
    GModel& G = ctx->G;
    G.loaded = false;
    release_refine(ctx->GR);
    G.blob.assign(blob, blob + n_floats);
    const float* p = blob;
    const float* lw = p; p += static_cast<size_t>(F) * nd;
    const float* lb = p; p += F;
    const float *g0 = p, *be0 = p + F, *m0 = p + 2 * static_cast<size_t>(F), *v0 = p + 3 * static_cast<size_t>(F); p += 4 * static_cast<size_t>(F);
    const float* w1 = p; p += 256u * 512 * 9;
    const float* b1 = p; p += 256;
    const float *g1 = p, *be1 = p + 256, *m1 = p + 512, *v1 = p + 768; p += 1024;
    const float* w2 = p; p += 128u * 256 * 9;
    const float* b2 = p; p += 128;
    const float *g2 = p, *be2 = p + 128, *m2 = p + 256, *v2 = p + 384; p += 512;
    const float* w3 = p; p += static_cast<size_t>(C) * 128 * 9;
    const float* b3 = p;

    G.C = C; G.H = H; G.W = W; G.nd = nd; G.F = F;
    G.cta_pairs = ctx->cta_pairs;
    const int pairs1 = (ctx->cta_pairs & 1) ? 2 : 1, pairs2 = (ctx->cta_pairs & 2) ? 2 : 1;
    G.kpad = (nd + 63) / 64 * 64;
    {   // Linear + BN1d + ReLU; output features re-ordered from View(512,sH,sW) (NCHW, models.lua:118) to NHWC
        std::vector<float> wm(static_cast<size_t>(F) * G.kpad, 0.0f);
        std::vector<float> bb(F), gg(F), be(F), mm(F), vv(F);
        for (int c = 0; c < 512; ++c)
            for (int s = 0; s < HW0; ++s) {
                const int fo = c * HW0 + s, fn = s * 512 + c;
                memcpy(&wm[static_cast<size_t>(fn) * G.kpad], lw + static_cast<size_t>(fo) * nd, sizeof(float) * nd);
                bb[fn] = lb[fo]; gg[fn] = g0[fo]; be[fn] = be0[fo]; mm[fn] = m0[fo]; vv[fn] = v0[fo];
            }
        BnFold bn = fold_bn(bb.data(), gg.data(), be.data(), mm.data(), vv.data(), F, F);
        const LayerDef d{"g_linear", KIND_LINEAR, 256, 1, 1, false, 1, 1, G.kpad, F, F / 256, 1, 1, F, 0, ACT_RELU, 1.0f, 0, false};
        RC_TRY(build_tc_layer(ctx, G.lin, d, wm.data(), bn));
    }
    {
        BnFold bn = fold_bn(b1, g1, be1, m1, v1, 256, 256);
        const LayerDef d{"g_conv1_up", KIND_UPCONV3, 256, pairs1 == 2 ? 1 : 2, pairs1, false,   // pairs: one double-buffered accumulator per CTA, B shared by the pair
                          sH, sW, 512, 256, 1, 2 * sH, 2 * sW, 256, 0, ACT_RELU, 1.0f, 0, false};
        RC_TRY(build_tc_layer(ctx, G.c1, d, w1, bn));
    }
    {
        BnFold bn = fold_bn(b2, g2, be2, m2, v2, 128, 128);
        const LayerDef d{"g_conv2_up", KIND_UPCONV3, 128, 2, pairs2, false, 2 * sH, 2 * sW, 256, 128, 1, H, W, 128, 0, ACT_RELU, 1.0f, 0, false};
        RC_TRY(build_tc_layer(ctx, G.c2, d, w2, bn));
    }
    {   // conv3 (128 -> C) + Sigmoid in two passes: a 1x1 GEMM giving every input pixel's 9*C tap
        // products (N = 16 or 32 fp32 per pixel), then g_conv3_gather_kernel sums the 9 neighbours.
        const int NT3 = C == 1 ? 16 : 32;
        std::vector<float> wm(static_cast<size_t>(NT3) * 128, 0.0f);
        for (int t = 0; t < 9; ++t)
            for (int co = 0; co < C; ++co)
                for (int ci = 0; ci < 128; ++ci) wm[static_cast<size_t>(t * C + co) * 128 + ci] = w3[(static_cast<size_t>(co) * 128 + ci) * 9 + t];
        BnFold bn;
        bn.scale.assign(NT3, 1.0f); bn.shift.assign(NT3, 0.0f);
        const LayerDef d{"g_conv3_taps", KIND_LINEAR, NT3, 1, 1, false, 1, 1, 128, 9 * C, 1, 1, 1, NT3, 0, ACT_NONE, 1.0f, 1, false};
        RC_TRY(build_tc_layer(ctx, G.c3, d, wm.data(), bn));
        RC_TRY(upload(ctx, G.b3, b3, sizeof(float) * C));
        // fused form (conv2 must be one of the MT = 2 variants): (tap, channel)-major fp32 weights for conv2's epilogue
        G.fuse3 = (ctx->fuse_conv3 == 2 || (ctx->fuse_conv3 == 1 && C == 1)) && G.c2.NT == 128 && G.c2.MT == 2;
        if (G.fuse3) {
            std::vector<float> wt(static_cast<size_t>(9) * C * 128);
            for (int t = 0; t < 9; ++t)
                for (int co = 0; co < C; ++co)
                    for (int ci = 0; ci < 128; ++ci) wt[static_cast<size_t>(t * C + co) * 128 + ci] = w3[(static_cast<size_t>(co) * 128 + ci) * 9 + t];
            RC_TRY(upload(ctx, G.w3f, wt.data(), sizeof(float) * wt.size()));
        }
    }
    G.loaded = true;
    return GANREV_OK;
}

static int load_R_impl(ganrev_ctx* ctx, int slot, int C, int H, int W, int nd, int tanh_out, const float* blob, size_t n_floats) {
    RC_TRY(check_geom(ctx, C, H, W, nd));
    if (slot < 0 || slot > 1) return fail(ctx, GANREV_EINVAL, "slot must be 0 or 1");
    const int Hh = H / 2, Wh = W / 2, Hq = H / 4, Wq = W / 4, HWq = Hq * Wq, F = 128 * HWq;
    const size_t need = static_cast<size_t>(64) * C * 9 + 5 * 64 + 2 * (64u * 64 * 9 + 5 * 64) + (128u * 64 * 9 + 5 * 128) +
                        2 * (128u * 128 * 9 + 5 * 128) + 512 * static_cast<size_t>(F) + 5 * 512 + static_cast<size_t>(nd) * 512 + nd;
    if (n_floats != need) return fail(ctx, GANREV_EINVAL, "R blob has %zu floats, expected %zu", n_floats, need);
    adopt_geometry(ctx, C, H, W, nd);
    RModel& R = ctx->R[slot];
    R.loaded = false;
    R.C = C; R.H = H; R.W = W; R.nd = nd; R.tanh_out = tanh_out;
    const float* p = blob;
    struct CB { const float *w, *b, *g, *be, *m, *v; };
    auto take_cb = [&](int co, int ci) {
        CB c;
        c.w = p; p += static_cast<size_t>(co) * ci * 9;
        c.b = p; p += co;
        c.g = p; c.be = p + co; c.m = p + 2 * co; c.v = p + 3 * co; p += 4 * co;
        return c;
    };
    const CB c1 = take_cb(64, C), c2 = take_cb(64, 64), c3 = take_cb(64, 64), c4 = take_cb(128, 64), c5 = take_cb(128, 128), c6 = take_cb(128, 128);
    const float* l1w = p; p += 512 * static_cast<size_t>(F);
    const float* l1b = p; p += 512;
    const float *g7 = p, *be7 = p + 512, *m7 = p + 1024, *v7 = p + 1536; p += 2048;
    const float* l2w = p; p += static_cast<size_t>(nd) * 512;
    const float* l2b = p;

    {   // conv1 pack: [k=(ci*3+ky)*3+kx][64] + scale[64] + shift[64]
        const int K = C * 9;
        std::vector<float> pack(static_cast<size_t>(K) * 64 + 128);
        for (int co = 0; co < 64; ++co)
            for (int k = 0; k < K; ++k) pack[static_cast<size_t>(k) * 64 + co] = c1.w[static_cast<size_t>(co) * K + k];
        BnFold bn = fold_bn(c1.b, c1.g, c1.be, c1.m, c1.v, 64, 64);
        memcpy(&pack[static_cast<size_t>(K) * 64], bn.scale.data(), 64 * 4);
        memcpy(&pack[static_cast<size_t>(K) * 64 + 64], bn.shift.data(), 64 * 4);
        RC_TRY(upload(ctx, R.c1pack, pack.data(), pack.size() * 4));
        // tcgen05 conv1 (conv1_tc.cuh): K index k = (ci*3+ky)*3+kx for the bf16 hi part of a tap, K + k for its lo part
        const int KP = C == 1 ? 32 : 64;
        std::vector<uint16_t> wb(static_cast<size_t>(64) * KP, 0);
        for (int co = 0; co < 64; ++co)
            for (int k = 0; k < K; ++k) wb[static_cast<size_t>(co) * KP + k] = wb[static_cast<size_t>(co) * KP + K + k] = f2bf(c1.w[static_cast<size_t>(co) * K + k] * bn.scale[co]);
        RC_TRY(upload(ctx, R.c1w, wb.data(), wb.size() * 2));
        RC_TRY(upload(ctx, R.c1shift, bn.shift.data(), 64 * 4));
    }
    auto conv_layer = [&](TcLayer& L, const char* name, const CB& c, int co, int ci, int Hin, int Win, int pool, float post, int MT, bool bres, int pairs) {
        BnFold bn = fold_bn(c.b, c.g, c.be, c.m, c.v, co, co);
        const int Ho = pool ? Hin / 2 : Hin, Wo = pool ? Win / 2 : Win;
        const LayerDef d{name, KIND_CONV3, co, MT, pairs, bres, Hin, Win, ci, co, 1, Ho, Wo, co, pool, ACT_ELU, post, 0, false};
        return build_tc_layer(ctx, L, d, c.w, bn);
    };
    // 64-channel layers: an item of MT = 2 sub-tiles is 72 MMAs (~2900 cycles) against ~900 cycles of accumulator / stage hand-off
    // (DESIGN section 6 finding 9); MT = 4 (cta_pairs bit 5, CTA pairs only: half of B per CTA leaves the room) amortises it over 144
    const int mt64 = ((ctx->cta_pairs & 4) && (ctx->cta_pairs & 32) && H * W >= 128 && W >= 8) ? 4 : 2;
    RC_TRY(conv_layer(R.c2, "r_conv2", c2, 64, 64, H, W, 0, 1.0f, mt64, true, (ctx->cta_pairs & 4) ? 2 : 1));
    RC_TRY(conv_layer(R.c3, "r_conv3_pool", c3, 64, 64, H, W, 1, 1.0f, mt64, true, (ctx->cta_pairs & 4) ? 2 : 1));
    const bool c4_pairs = (ctx->cta_pairs & 8) && Hh * Wh >= 128 && Wh >= 8;   // CTA pairs exist for the halo-reuse tiling only
    RC_TRY(conv_layer(R.c4, "r_conv4", c4, 128, 64, Hh, Wh, 0, 1.0f, c4_pairs ? 2 : 1, true, (ctx->cta_pairs & 8) ? 2 : 1));   // pairs: half of B per CTA leaves room for MT = 2
    RC_TRY(conv_layer(R.c5, "r_conv5", c5, 128, 128, Hh, Wh, 0, 1.0f, 2, false, (ctx->cta_pairs & 16) ? 2 : 1));
    RC_TRY(conv_layer(R.c6, "r_conv6_pool", c6, 128, 128, Hh, Wh, 1, 1.0f, 2, false, (ctx->cta_pairs & 16) ? 2 : 1));   // its SpatialDropout(0.25) x0.75 is folded into r_linear1
    {   // Linear(F -> 512) + BN1d + ELU; input columns re-ordered from View (NCHW flatten, models.lua:446) to NHWC.
        // The eval-mode SpatialDropout(0.25) in front of it (y = 0.75 x, models.lua:439; it commutes with the max-pool after it) is linear, so it
        // is folded into these weights instead of costing a multiply per activation in conv6's epilogue.
        std::vector<float> wm(static_cast<size_t>(512) * F);
        for (int o = 0; o < 512; ++o)
            for (int c = 0; c < 128; ++c)
                for (int s = 0; s < HWq; ++s) wm[static_cast<size_t>(o) * F + s * 128 + c] = 0.75f * l1w[static_cast<size_t>(o) * F + c * HWq + s];
        BnFold bn = fold_bn(l1b, g7, be7, m7, v7, 512, 512);
        const LayerDef d{"r_linear1", KIND_LINEAR, 256, 1, 1, false, 1, 1, F, 512, 2, 1, 1, 512, 0, ACT_ELU, 1.0f, 0, false};   // N = 256: the A tile is re-read twice, not 8 times
        RC_TRY(build_tc_layer(ctx, R.l1, d, wm.data(), bn));
    }
    {   // Linear(512 -> nd) [+ Tanh], fp32 output
        const int NT = nd <= 32 ? 32 : (nd <= 64 ? 64 : (nd <= 128 ? 128 : 256));
        const int n_tiles = (nd + NT - 1) / NT, cp = n_tiles * NT;
        std::vector<float> wm(static_cast<size_t>(cp) * 512, 0.0f);
        memcpy(wm.data(), l2w, sizeof(float) * static_cast<size_t>(nd) * 512);
        BnFold bn;
        bn.scale.assign(cp, 0.0f); bn.shift.assign(cp, 0.0f);
        for (int i = 0; i < nd; ++i) { bn.scale[i] = 1.0f; bn.shift[i] = l2b[i]; }
        const LayerDef d{"r_linear2", KIND_LINEAR, NT, 1, 1, false, 1, 1, 512, nd, n_tiles, 1, 1, nd, 0, tanh_out ? ACT_TANH : ACT_NONE, 1.0f, 1, false};
        RC_TRY(build_tc_layer(ctx, R.l2, d, wm.data(), bn));
    }
    R.loaded = true;
    return GANREV_OK;
}

// =================================================================================
// pipelines (device pointers in, device pointers out)
// =================================================================================
// Images per chunk: every layer of a chunk is one kernel launch, and each launch pays a fixed ~15 us (launch gap, barrier /
// TMEM set-up, pipeline fill and drain, last-wave quantisation): measured 1.07 M img/s at 4096 32x32 faces per chunk, 1.13 M at
// 8192, flat beyond.  Auto = 8192 faces' worth of pixels (2 x 2 GB activation arenas at any geometry).
static int64_t chunk_for(const ganrev_ctx* ctx, int H, int W) {
    if (ctx->chunk > 0) return ctx->chunk;
    return std::max<int64_t>(256, (8192LL * 1024) / (static_cast<int64_t>(H) * W));
}
static int ensure_arena(ganrev_ctx* ctx, size_t per_img_bytes, int64_t chunk) {
    RC_TRY(ensure(ctx, ctx->arena[0], per_img_bytes * chunk));
    RC_TRY(ensure(ctx, ctx->arena[1], per_img_bytes * chunk));
    return GANREV_OK;
}

// Host <-> device copies of a chunked forward pass, overlapped with the kernels: every input chunk is copied on `copy_in` (an event
// per chunk, the compute stream waits for its chunk only), every output chunk goes back on `copy_out` as soon as its last kernel has
// finished.  With pageable host memory the copies are staged by the driver and simply do not overlap; results are identical.
struct ChunkIO {
    const uint8_t* h_in = nullptr;  uint8_t* d_in = nullptr;        size_t in_row = 0;    // one row = one image / noise vector
    uint8_t* h_out = nullptr;       const uint8_t* d_out = nullptr; size_t out_row = 0;
    int first_event = 0;
};
static int chunk_io_begin(ganrev_ctx* ctx, ChunkIO* io, int64_t N, int64_t CH) {
    if (!io || (!io->h_in && !io->h_out) || N <= 0) return GANREV_OK;
    if (!ctx->copy_in) {
        CU_TRY(cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
        CU_TRY(cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
    }
    const int64_t chunks = (N + CH - 1) / CH;
    while (static_cast<int64_t>(ctx->io_events.size()) < 2 * chunks + 1) {   // [0, chunks) inputs landed, [chunks, 2 chunks) outputs ready, [2 chunks] start
        cudaEvent_t e;
        CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->io_events.push_back(e);
    }
    ctx->copies_pending = true;
    if (io->h_in) {
        // the copy stream starts behind whatever the compute stream has queued so far (buffer growth, earlier readers of the buffer)
        cudaEvent_t e0 = ctx->io_events[2 * chunks];
        CU_TRY(cudaEventRecord(e0, ctx->stream));
        CU_TRY(cudaStreamWaitEvent(ctx->copy_in, e0, 0));
        for (int64_t c = 0; c < chunks; ++c) {
            const int64_t n0 = c * CH, n = std::min<int64_t>(CH, N - n0);
            CU_TRY(cudaMemcpyAsync(io->d_in + n0 * io->in_row, io->h_in + n0 * io->in_row, static_cast<size_t>(n) * io->in_row, cudaMemcpyHostToDevice, ctx->copy_in));
            CU_TRY(cudaEventRecord(ctx->io_events[c], ctx->copy_in));
        }
    }
    return GANREV_OK;
}
static int chunk_io_before(ganrev_ctx* ctx, const ChunkIO* io, int64_t c) {
    if (io && io->h_in) CU_TRY(cudaStreamWaitEvent(ctx->stream, ctx->io_events[c], 0));
    return GANREV_OK;
}
static int chunk_io_after(ganrev_ctx* ctx, const ChunkIO* io, int64_t c, int64_t chunks, int64_t n0, int64_t n) {
    if (io && io->h_out) {
        cudaEvent_t e = ctx->io_events[chunks + c];
        CU_TRY(cudaEventRecord(e, ctx->stream));
        CU_TRY(cudaStreamWaitEvent(ctx->copy_out, e, 0));
        CU_TRY(cudaMemcpyAsync(io->h_out + n0 * io->out_row, io->d_out + n0 * io->out_row, static_cast<size_t>(n) * io->out_row, cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    return GANREV_OK;
}

// Layers of forward_G_dev / forward_R_dev, in the order they run (ganrev_debug_G_stage / ganrev_debug_R_stage number them the same
// way).  GLAYER_C2 is G conv2's activation h2, which only exists when the tap products are not fused into conv2's epilogue.
enum { GLAYER_LIN = 0, GLAYER_C1, GLAYER_C2, GLAYER_TAPS, GLAYER_Y, GLAYER_COUNT };
enum { RLAYER_C1 = 0, RLAYER_C2, RLAYER_C3, RLAYER_C4, RLAYER_C5, RLAYER_C6, RLAYER_L1, RLAYER_OUT, RLAYER_COUNT };

// stop_after < GLAYER_Y (tests) returns once that layer's buffer is written; call it with N <= one chunk then, or the next chunk
// overwrites it.
static int forward_G_dev(ganrev_ctx* ctx, const float* d_noise, int64_t N, float* d_images, ChunkIO* io = nullptr, int stop_after = GLAYER_Y) {
    GModel& G = ctx->G;
    if (!G.loaded) return fail(ctx, GANREV_ESTATE, "G not loaded");
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, G.H, G.W), std::max<int64_t>(N, 1));
    const size_t per_img = static_cast<size_t>(G.H) * G.W * 128 * 2;   // largest activation (conv2 out); a0/a1 are smaller
    RC_TRY(ensure_arena(ctx, per_img, CH));
    RC_TRY(ensure(ctx, ctx->noise_bf16, static_cast<size_t>(CH) * G.kpad * 2));
    RC_TRY(chunk_io_begin(ctx, io, N, CH));
    const int64_t n_chunks = (N + CH - 1) / CH;
    for (int64_t n0 = 0; n0 < N; n0 += CH) {
        const int n = static_cast<int>(std::min<int64_t>(CH, N - n0));
        RC_TRY(chunk_io_before(ctx, io, n0 / CH));
        {
            ProfScope ps(ctx, "g_noise_to_bf16", 0.0, static_cast<double>(n) * (G.nd * 4.0 + G.kpad * 2.0));
            const long long tot = static_cast<long long>(n) * G.kpad;
            noise_to_bf16_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, ctx->stream>>>(
                d_noise + n0 * G.nd, G.nd, G.kpad, reinterpret_cast<bf16*>(ctx->noise_bf16.p), n);
            CU_TRY(cudaGetLastError());
        }
        RC_TRY(run_layer(ctx, G.lin, ctx->noise_bf16.p, ctx->arena[0].p, n, CH));   // [n][sH][sW][512]
        if (stop_after == GLAYER_LIN) return GANREV_OK;
        RC_TRY(run_layer(ctx, G.c1, ctx->arena[0].p, ctx->arena[1].p, n, CH));      // [n][2sH][2sW][256]
        if (stop_after == GLAYER_C1) return GANREV_OK;
        // tap products of the last conv as 9*C planes of `plane` floats, P[tap*C + co][pixel]: stores and the gather's loads
        // are then contiguous per warp, and zero-padded columns are never written
        const long long plane = static_cast<long long>(CH) * G.H * G.W;
        const bool fused = G.fuse3 && ctx->conv_impl == 0;
        G.c2.g.w3 = fused ? static_cast<const float*>(G.w3f.p) : nullptr;
        G.c2.g.w3_c = G.C;
        G.c2.g.taps = static_cast<float*>(ctx->arena[0].p);
        G.c2.g.taps_plane = plane;
        RC_TRY(run_layer(ctx, G.c2, ctx->arena[1].p, ctx->arena[0].p, n, CH));      // [n][H][W][128], or (fused) the tap planes
        if (stop_after == GLAYER_C2) return GANREV_OK;
        {   // last conv: per-pixel tap products (conv2's epilogue, or a 1x1 GEMM on the tensor cores), then the 3x3 gather + bias + sigmoid
            const long long npix = static_cast<long long>(n) * G.H * G.W;
            const float* planes = static_cast<const float*>(ctx->arena[fused ? 0 : 1].p);
            if (!fused) {
                G.c3.g.out_sN = 1; G.c3.g.out_sP = 1; G.c3.g.out_sC = static_cast<int>(plane);
                G.c3.bytes_per_img = 2.0 * 128 + 4.0 * 9 * G.C;
                RC_TRY(run_layer(ctx, G.c3, ctx->arena[0].p, ctx->arena[1].p, static_cast<int>(npix), CH * G.H * G.W));
            }
            if (stop_after == GLAYER_TAPS) return GANREV_OK;
            ProfScope ps(ctx, "g_conv3_gather", 9.0 * npix * G.C, npix * (4.0 * 9 * G.C + 4.0 * G.C));
            const unsigned blocks = static_cast<unsigned>((npix / 4 + 255) / 256);      // a thread per 4 pixels of a row (W >= 16, a power of two)
            float* o = d_images + n0 * G.C * G.H * G.W;
            if (G.C == 1) g_conv3_gather_kernel<1><<<blocks, 256, 0, ctx->stream>>>(planes, plane, static_cast<const float*>(G.b3.p), o, G.H, G.W, ilog2(G.H), ilog2(G.W), n);
            else          g_conv3_gather_kernel<3><<<blocks, 256, 0, ctx->stream>>>(planes, plane, static_cast<const float*>(G.b3.p), o, G.H, G.W, ilog2(G.H), ilog2(G.W), n);
            CU_TRY(cudaGetLastError());
        }
        RC_TRY(chunk_io_after(ctx, io, n0 / CH, n_chunks, n0, n));
    }
    return GANREV_OK;
}

// stop_after < RLAYER_OUT (tests): as forward_G_dev.
static int forward_R_dev(ganrev_ctx* ctx, int slot, const float* d_images, const uint8_t* d_mask, int64_t N, float* d_attrs, ChunkIO* io = nullptr,
                         int stop_after = RLAYER_OUT) {
    if (slot < 0 || slot > 1) return fail(ctx, GANREV_EINVAL, "slot must be 0 or 1");
    RModel& R = ctx->R[slot];
    if (!R.loaded) return fail(ctx, GANREV_ESTATE, "R slot %d not loaded", slot);
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, R.H, R.W), std::max<int64_t>(N, 1));
    const size_t per_img = static_cast<size_t>(R.H) * R.W * 64 * 2;   // conv1/conv2 outputs are the largest
    RC_TRY(ensure_arena(ctx, per_img, CH));
    const long long img_elems = static_cast<long long>(R.C) * R.H * R.W;
    RC_TRY(chunk_io_begin(ctx, io, N, CH));
    const int64_t n_chunks = (N + CH - 1) / CH;
    for (int64_t n0 = 0; n0 < N; n0 += CH) {
        const int n = static_cast<int>(std::min<int64_t>(CH, N - n0));
        RC_TRY(chunk_io_before(ctx, io, n0 / CH));
        {
            const long long npix = static_cast<long long>(n) * R.H * R.W;
            ProfScope ps(ctx, "r_conv1", 2.0 * npix * 64 * 9 * R.C, npix * (R.C * (4.0 + (d_mask ? 1.0 : 0.0)) + 128.0));
            const unsigned blocks = static_cast<unsigned>((npix + 127) / 128);
            const float* in = d_images + n0 * img_elems;
            const uint8_t* mk = d_mask ? d_mask + n0 * img_elems : nullptr;
            if (ctx->conv_impl == 0) {
                const int n_tiles = static_cast<int>(blocks);
                // resident CTAs per SM: bounded by registers (128 threads each) and 512 TMEM columns / 64; shared memory
                // (26 KB each) is not the limit once the carve-out favours it.  One even wave of persistent CTAs.
                static int occ_dev[kMaxDevices][2] = {};
                int& occ = occ_dev[ctx->device][R.C == 1 ? 0 : 1];
                if (occ == 0) {
                    cudaFuncAttributes fa{};
                    if (R.C == 1) { CU_TRY(cudaFuncGetAttributes(&fa, tc::r_conv1_tc_kernel<1>)); CU_TRY(cudaFuncSetAttribute(tc::r_conv1_tc_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); }
                    else          { CU_TRY(cudaFuncGetAttributes(&fa, tc::r_conv1_tc_kernel<3>)); CU_TRY(cudaFuncSetAttribute(tc::r_conv1_tc_kernel<3>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); }
                    const int regs = ((std::max(fa.numRegs, 32) + 7) / 8) * 8;
                    occ = std::max(1, std::min(8, 65536 / (128 * regs)));
                }
                const int grid = std::min(n_tiles, ctx->num_sms * occ);
                const int lgW = ilog2(R.W), lgHW = ilog2(R.H * R.W);
                if (R.C == 1)
                    tc::r_conv1_tc_kernel<1><<<grid, 128, tc::Conv1Cfg<1>::kSmemBytes, ctx->stream>>>(in, mk, reinterpret_cast<const bf16*>(R.c1w.p), reinterpret_cast<const float*>(R.c1shift.p),
                        reinterpret_cast<bf16*>(ctx->arena[0].p), R.H, R.W, lgW, lgHW, npix, n_tiles, ctx->d_err_flag);
                else
                    tc::r_conv1_tc_kernel<3><<<grid, 128, tc::Conv1Cfg<3>::kSmemBytes, ctx->stream>>>(in, mk, reinterpret_cast<const bf16*>(R.c1w.p), reinterpret_cast<const float*>(R.c1shift.p),
                        reinterpret_cast<bf16*>(ctx->arena[0].p), R.H, R.W, lgW, lgHW, npix, n_tiles, ctx->d_err_flag);
            } else if (R.C == 1)
                r_conv1_kernel<1><<<blocks, 128, 0, ctx->stream>>>(in, mk, (const float*)R.c1pack.p, reinterpret_cast<bf16*>(ctx->arena[0].p), R.H, R.W, npix);
            else
                r_conv1_kernel<3><<<blocks, 128, 0, ctx->stream>>>(in, mk, (const float*)R.c1pack.p, reinterpret_cast<bf16*>(ctx->arena[0].p), R.H, R.W, npix);
            CU_TRY(cudaGetLastError());
        }
        if (stop_after == RLAYER_C1) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.c2, ctx->arena[0].p, ctx->arena[1].p, n, CH));
        if (stop_after == RLAYER_C2) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.c3, ctx->arena[1].p, ctx->arena[0].p, n, CH));
        if (stop_after == RLAYER_C3) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.c4, ctx->arena[0].p, ctx->arena[1].p, n, CH));
        if (stop_after == RLAYER_C4) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.c5, ctx->arena[1].p, ctx->arena[0].p, n, CH));
        if (stop_after == RLAYER_C5) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.c6, ctx->arena[0].p, ctx->arena[1].p, n, CH));
        if (stop_after == RLAYER_C6) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.l1, ctx->arena[1].p, ctx->arena[0].p, n, CH));
        if (stop_after == RLAYER_L1) return GANREV_OK;
        RC_TRY(run_layer(ctx, R.l2, ctx->arena[0].p, d_attrs + n0 * R.nd, n, CH));
        RC_TRY(chunk_io_after(ctx, io, n0 / CH, n_chunks, n0, n));
    }
    return GANREV_OK;
}

static int l2_dev(ganrev_ctx* ctx, const float* a, const float* b, int64_t N, int px, double* out) {
    ProfScope ps(ctx, "l2_pairs", 3.0 * N * px, 8.0 * N * px + 8.0 * N);
    const unsigned blocks = static_cast<unsigned>((N * 32 + 255) / 256);
    if (N > 0) l2_pairs_kernel<<<blocks, 256, 0, ctx->stream>>>(a, b, N, px, out);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}


// ---------------------------------------------------------------- noise-vector refinement (DESIGN.md section 4.5)
// G's backward layers, from the host copy of the blob.  With BN folded (s = scale): conv^T is a plain 3x3 conv at the high
// resolution with weights W^T[ci][2-ky][2-kx][co] * s[co]; the 2x2 sum-pool (adjoint of nearest upsampling) and the ReLU mask of
// the stored forward activation are the MASKSUM epilogue; Linear^T is the K = F GEMM in the forward's NHWC feature order with s0
// folded.  N = 128 tiles: a 256-wide tile with halo reuse needs 116 KB per pipeline unit, two stages do not fit in shared memory.
static int build_refine(ganrev_ctx* ctx) {
    GRefine& R = ctx->GR;
    if (R.built) return GANREV_OK;
    const GModel& G = ctx->G;
    const int C = G.C, H = G.H, W = G.W, nd = G.nd, HW0 = (H / 4) * (W / 4), F = G.F;
    const float* p = G.blob.data();
    const float* lw = p; p += static_cast<size_t>(F) * nd;
    p += F;                                                                  // Linear bias (in the forward's shift only)
    const float *g0 = p, *v0 = p + 3 * static_cast<size_t>(F); p += 4 * static_cast<size_t>(F);
    const float* w1 = p; p += 256u * 512 * 9 + 256;
    const float *g1 = p, *v1 = p + 768; p += 1024;
    const float* w2 = p; p += 128u * 256 * 9 + 128;
    const float *g2 = p, *v2 = p + 384; p += 512;
    const float* w3 = p;
    auto sc = [](const float* g, const float* v, size_t i) { return g[i] / std::sqrt(v[i] + 1e-5f); };   // fold_bn's scale
    const int pairs = (G.cta_pairs & 16) ? 2 : 1;      // the pooled 128-wide tile of R conv6 (same kernel shape); cta_pairs as at load_G
    auto conv_t = [&](TcLayer& L, const char* name, const float* w, const float* g, const float* v, int co_f, int ci_f, int Hin, int Win) {
        // forward conv ci_f -> co_f; adjoint co_f -> ci_f at the forward conv's (high) resolution, pooled to the forward input's
        std::vector<float> wt(static_cast<size_t>(ci_f) * co_f * 9);
        for (int b = 0; b < co_f; ++b) {
            const float s = sc(g, v, b);
            for (int a = 0; a < ci_f; ++a)
                for (int t = 0; t < 9; ++t) wt[(static_cast<size_t>(a) * co_f + b) * 9 + t] = w[(static_cast<size_t>(b) * ci_f + a) * 9 + (8 - t)] * s;
        }
        BnFold one;
        one.scale.assign(ci_f, 1.0f); one.shift.assign(ci_f, 0.0f);
        const LayerDef d{name, KIND_CONV3, 128, 2, pairs, false, Hin, Win, co_f, ci_f, ci_f / 128, Hin / 2, Win / 2, ci_f, 1, ACT_NONE, 1.0f, 0, false};
        return build_tc_layer(ctx, L, d, wt.data(), one);
    };
    RC_TRY(conv_t(R.c2t, "g_bwd_conv2", w2, g2, v2, 128, 256, H, W));
    RC_TRY(conv_t(R.c1t, "g_bwd_conv1", w1, g1, v1, 256, 512, H / 2, W / 2));
    {   // Linear^T: [nd (padded)][F], column fn = s*512 + c (NHWC) <- forward row fo = c*HW0 + s (View(512, sH, sW))
        const int NT = nd <= 32 ? 32 : (nd <= 64 ? 64 : (nd <= 128 ? 128 : 256));
        const int n_tiles = (nd + NT - 1) / NT, cp = n_tiles * NT;
        std::vector<float> wm(static_cast<size_t>(cp) * F, 0.0f);
        for (int c = 0; c < 512; ++c)
            for (int s = 0; s < HW0; ++s) {
                const size_t fo = static_cast<size_t>(c) * HW0 + s, fn = static_cast<size_t>(s) * 512 + c;
                const float s0 = sc(g0, v0, fo);
                for (int k = 0; k < nd; ++k) wm[static_cast<size_t>(k) * F + fn] = lw[fo * nd + k] * s0;
            }
        BnFold bn;
        bn.scale.assign(cp, 0.0f); bn.shift.assign(cp, 0.0f);
        for (int i = 0; i < nd; ++i) bn.scale[i] = 1.0f;
        const LayerDef d{"g_bwd_linear", KIND_LINEAR, NT, 1, 1, false, 1, 1, F, nd, n_tiles, 1, 1, nd, 0, ACT_NONE, 1.0f, 1, false};
        RC_TRY(build_tc_layer(ctx, R.lint, d, wm.data(), bn));
    }
    std::vector<float> w3t(static_cast<size_t>(9) * C * 128);
    for (int t = 0; t < 9; ++t)
        for (int co = 0; co < C; ++co)
            for (int ci = 0; ci < 128; ++ci) w3t[(static_cast<size_t>(t) * C + co) * 128 + ci] = w3[(static_cast<size_t>(co) * 128 + ci) * 9 + t];
    RC_TRY(upload(ctx, R.w3t, w3t.data(), w3t.size() * 4));
    R.built = true;
    return GANREV_OK;
}

static int refine_buffers(ganrev_ctx* ctx, int64_t CH) {
    const GModel& G = ctx->G;
    GRefine& R = ctx->GR;
    const size_t px = static_cast<size_t>(G.H) * G.W;
    RC_TRY(ensure_arena(ctx, px * 128 * 2, CH));   // e2 (the largest gradient), then e0; e1 and the last conv's tap planes in the other
    RC_TRY(ensure(ctx, ctx->noise_bf16, static_cast<size_t>(CH) * G.kpad * 2));
    RC_TRY(ensure(ctx, R.h0, static_cast<size_t>(CH) * G.F * 2));
    RC_TRY(ensure(ctx, R.h1, static_cast<size_t>(CH) * px / 4 * 256 * 2));
    RC_TRY(ensure(ctx, R.h2, static_cast<size_t>(CH) * px * 128 * 2));
    RC_TRY(ensure(ctx, R.y, static_cast<size_t>(CH) * G.C * px * 4));
    for (DevBuf* b : {&R.glin, &R.m, &R.v}) RC_TRY(ensure(ctx, *b, static_cast<size_t>(CH) * G.nd * 4));
    return GANREV_OK;
}

// Stages of refine_grad_chunk, in the order it produces them (ganrev_debug_refine_stage numbers them the same way)
enum { RSTAGE_H0 = 0, RSTAGE_H1, RSTAGE_H2, RSTAGE_Y, RSTAGE_E2, RSTAGE_E1, RSTAGE_E0, RSTAGE_GLIN, RSTAGE_COUNT };

// One forward pass of G keeping h0 / h1 / h2 (bf16 NHWC) and y = G(z) (fp32 NCHW, in R.y), then the backward pass down to
// R.glin[n x nd] = W_lin^T (s0 e0), the gradient of ||G(z) - x||^2 without the prior term.  n <= CH images.  stop_after < RSTAGE_GLIN
// (tests) returns once that stage's buffer is written: conv1^T writes e0 over e2 in arena[0].
static int refine_grad_chunk(ganrev_ctx* ctx, const float* d_z, const float* d_x, int n, int64_t CH, int stop_after = RSTAGE_GLIN) {
    GModel& G = ctx->G;
    GRefine& R = ctx->GR;
    const int H = G.H, W = G.W;
    const long long npix = static_cast<long long>(n) * H * W, plane = static_cast<long long>(CH) * H * W;
    {
        ProfScope ps(ctx, "g_noise_to_bf16", 0.0, static_cast<double>(n) * (G.nd * 4.0 + G.kpad * 2.0));
        const long long tot = static_cast<long long>(n) * G.kpad;
        noise_to_bf16_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, ctx->stream>>>(d_z, G.nd, G.kpad, reinterpret_cast<bf16*>(ctx->noise_bf16.p), n);
        CU_TRY(cudaGetLastError());
    }
    RC_TRY(run_layer(ctx, G.lin, ctx->noise_bf16.p, R.h0.p, n, CH));
    if (stop_after == RSTAGE_H0) return GANREV_OK;
    RC_TRY(run_layer(ctx, G.c1, R.h0.p, R.h1.p, n, CH));
    if (stop_after == RSTAGE_H1) return GANREV_OK;
    G.c2.g.w3 = nullptr;                                                        // unfused: h2 itself is needed
    RC_TRY(run_layer(ctx, G.c2, R.h1.p, R.h2.p, n, CH));
    if (stop_after == RSTAGE_H2) return GANREV_OK;
    G.c3.g.out_sN = 1; G.c3.g.out_sP = 1; G.c3.g.out_sC = static_cast<int>(plane);
    G.c3.bytes_per_img = 2.0 * 128 + 4.0 * 9 * G.C;
    RC_TRY(run_layer(ctx, G.c3, R.h2.p, ctx->arena[1].p, static_cast<int>(npix), CH * H * W));
    float* y = static_cast<float*>(R.y.p);
    {
        ProfScope ps(ctx, "g_conv3_gather", 9.0 * npix * G.C, npix * (4.0 * 9 * G.C + 4.0 * G.C));
        const unsigned blocks = static_cast<unsigned>((npix / 4 + 255) / 256);
        const float* planes = static_cast<const float*>(ctx->arena[1].p);
        if (G.C == 1) g_conv3_gather_kernel<1><<<blocks, 256, 0, ctx->stream>>>(planes, plane, static_cast<const float*>(G.b3.p), y, H, W, ilog2(H), ilog2(W), n);
        else          g_conv3_gather_kernel<3><<<blocks, 256, 0, ctx->stream>>>(planes, plane, static_cast<const float*>(G.b3.p), y, H, W, ilog2(H), ilog2(W), n);
        CU_TRY(cudaGetLastError());
    }
    if (stop_after == RSTAGE_Y) return GANREV_OK;
    bf16* e2 = static_cast<bf16*>(ctx->arena[0].p);
    {   // per pixel: 9*C taps into 128 channels; reads y, x (9*C neighbours, cached) and h2, writes e2
        ProfScope ps(ctx, "g_bwd_conv3", 2.0 * npix * 9 * G.C * 128, npix * (2.0 * 4 * G.C + 2.0 * 128 + 2.0 * 128));
        const unsigned blocks = static_cast<unsigned>((npix * 16 + 255) / 256);
        const bf16* h2 = static_cast<const bf16*>(R.h2.p);
        const float* w3t = static_cast<const float*>(R.w3t.p);
        if (G.C == 1) g_conv3_adjoint_kernel<1><<<blocks, 256, 0, ctx->stream>>>(y, d_x, w3t, h2, e2, H, W, ilog2(H), ilog2(W), n);
        else          g_conv3_adjoint_kernel<3><<<blocks, 256, 0, ctx->stream>>>(y, d_x, w3t, h2, e2, H, W, ilog2(H), ilog2(W), n);
        CU_TRY(cudaGetLastError());
    }
    if (stop_after == RSTAGE_E2) return GANREV_OK;
    R.c2t.g.ref = static_cast<const bf16*>(R.h1.p);
    RC_TRY(run_layer(ctx, R.c2t, e2, ctx->arena[1].p, n, CH));                  // e1 = [h1 > 0] * sumpool(conv2^T(e2))
    if (stop_after == RSTAGE_E1) return GANREV_OK;
    R.c1t.g.ref = static_cast<const bf16*>(R.h0.p);
    RC_TRY(run_layer(ctx, R.c1t, ctx->arena[1].p, ctx->arena[0].p, n, CH));     // e0 = [h0 > 0] * sumpool(conv1^T(e1))
    if (stop_after == RSTAGE_E0) return GANREV_OK;
    RC_TRY(run_layer(ctx, R.lint, ctx->arena[0].p, R.glin.p, n, CH));           // W_lin^T (s0 e0)
    return GANREV_OK;
}

// `iters` Adam steps on every row of d_z [N x nd] (in place).  Chunks run one after another, all iterations of a chunk at a time:
// nothing mixes images, so results do not depend on the chunk size or on which images share a call.
static int refine_dev(ganrev_ctx* ctx, const float* d_x, float* d_z, int64_t N, int iters, const float* hyper6) {
    GModel& G = ctx->G;
    GRefine& R = ctx->GR;
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, G.H, G.W), std::max<int64_t>(N, 1));
    RC_TRY(build_refine(ctx));
    RC_TRY(refine_buffers(ctx, CH));
    const long long px = static_cast<long long>(G.C) * G.H * G.W;
    for (int64_t n0 = 0; n0 < N; n0 += CH) {
        const int n = static_cast<int>(std::min<int64_t>(CH, N - n0));
        const long long ne = static_cast<long long>(n) * G.nd;
        float* z = d_z + n0 * G.nd;
        CU_TRY(cudaMemsetAsync(R.m.p, 0, sizeof(float) * ne, ctx->stream));
        CU_TRY(cudaMemsetAsync(R.v.p, 0, sizeof(float) * ne, ctx->stream));
        for (int t = 1; t <= iters; ++t) {
            RC_TRY(refine_grad_chunk(ctx, z, d_x + n0 * px, n, CH));
            RefineHyper h{};
            h.beta1 = hyper6[1]; h.beta2 = hyper6[2]; h.eps = hyper6[3]; h.prior2 = 2.0f * hyper6[4]; h.zclamp = hyper6[5];
            h.step_size = static_cast<float>(static_cast<double>(hyper6[0]) * std::sqrt(1.0 - std::pow(static_cast<double>(h.beta2), static_cast<double>(t))) /
                                             (1.0 - std::pow(static_cast<double>(h.beta1), static_cast<double>(t))));
            ProfScope ps(ctx, "refine_adam", 12.0 * ne, 24.0 * ne);
            refine_adam_kernel<<<static_cast<unsigned>((ne + 255) / 256), 256, 0, ctx->stream>>>(z, static_cast<const float*>(R.glin.p), static_cast<float*>(R.m.p), static_cast<float*>(R.v.p), ne, h);
            CU_TRY(cudaGetLastError());
        }
    }
    return GANREV_OK;
}

// =================================================================================
// C ABI
// =================================================================================
extern "C" {

int ganrev_version(void) { return 100; }

int ganrev_create(ganrev_ctx** out, int device) {
    if (!out) return GANREV_EINVAL;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return GANREV_ENODEV;
    if (device < 0 || device >= count || device >= kMaxDevices) return GANREV_ENODEV;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return GANREV_ENODEV;
    if (prop.major != 10) return GANREV_ENODEV;   // tcgen05 / TMEM kernels are sm_100a only; there is no fallback
    if (cudaSetDevice(device) != cudaSuccess) return GANREV_ECUDA;
    ganrev_ctx* ctx = new ganrev_ctx();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    int rc = GANREV_OK;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { ctx->stream = nullptr; rc = GANREV_ECUDA; }
    else if (cudaMalloc(&ctx->d_err_flag, sizeof(int)) != cudaSuccess) { ctx->d_err_flag = nullptr; rc = GANREV_ENOMEM; }
    else if (cudaMemset(ctx->d_err_flag, 0, sizeof(int)) != cudaSuccess) rc = GANREV_ECUDA;
    else if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) rc = GANREV_ECUDA;
    if (rc != GANREV_OK) {   // nothing created above outlives a failed create
        if (ctx->d_err_flag) cudaFree(ctx->d_err_flag);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return rc;
    }
    ctx->encode = reinterpret_cast<EncodeTiledFn>(fn);
    *out = ctx;
    return GANREV_OK;
}

void ganrev_destroy(ganrev_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    prof_resolve(ctx);
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->comm && ctx->nccl.CommDestroy) ctx->nccl.CommDestroy(ctx->comm);
    for (TcLayer* L : {&ctx->G.lin, &ctx->G.c1, &ctx->G.c2, &ctx->G.c3}) release_layer(*L);
    release(ctx->G.b3);
    release(ctx->G.w3f);
    release_refine(ctx->GR);
    for (int s = 0; s < 2; ++s) {
        RModel& R = ctx->R[s];
        release(R.c1pack); release(R.c1w); release(R.c1shift);
        for (TcLayer* L : {&R.c2, &R.c3, &R.c4, &R.c5, &R.c6, &R.l1, &R.l2}) release_layer(*L);
    }
    for (auto& b : ctx->buf) release(b);
    for (DevBuf* b : {&ctx->train.P, &ctx->train.Gd, &ctx->train.M, &ctx->train.V, &ctx->train.flags, &ctx->train.work, &ctx->train.masks, &ctx->train.partial, &ctx->train.lossbuf}) release(*b);
    for (DevBuf* b : {&ctx->nn_partial, &ctx->nn_ids, &ctx->nn_dist, &ctx->nn_flag, &ctx->nn_all, &ctx->qsel, &ctx->shard, &ctx->tfs_aux, &ctx->amb, &ctx->pdb, &ctx->pq, &ctx->tc_thr,
                      &ctx->tc_cnt, &ctx->tc_cand, &ctx->tc_pairs, &ctx->tc_keys, &ctx->tc_special, &ctx->tc_flags, &ctx->tc_dump}) release(*b);
    for (DevBuf* b : {&ctx->arena[0], &ctx->arena[1], &ctx->noise_bf16, &ctx->stage_a, &ctx->stage_b, &ctx->l2buf, &ctx->thr, &ctx->flags,
                      &ctx->db, &ctx->rdb, &ctx->maxabs, &ctx->q, &ctx->rq, &ctx->c2, &ctx->partial, &ctx->keys, &ctx->keys_all, &ctx->ids,
                      &ctx->scores, &ctx->cen, &ctx->acc, &ctx->cnt, &ctx->total, &ctx->labels, &ctx->cosv, &ctx->tcounts, &ctx->mids,
                      &ctx->mcnt, &ctx->mmean, &ctx->trace})
        release(*b);
    if (ctx->d_err_flag) cudaFree(ctx->d_err_flag);
    for (auto e : ctx->io_events) cudaEventDestroy(e);
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* ganrev_last_error(const ganrev_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

// ---------------------------------------------------------------- NCCL (dlopen)
static int nccl_load(ganrev_ctx* ctx) {
    NcclApi& a = ctx->nccl;
    if (a.h) return GANREV_OK;
    a.h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!a.h) a.h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!a.h) return fail(ctx, GANREV_ENCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
#define NCCL_SYM(field, sym)                                                     \
    a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.h, sym));              \
    if (!a.field) return fail(ctx, GANREV_ENCCL, "libnccl lacks %s", sym);
    NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    NCCL_SYM(CommInitRank, "ncclCommInitRank")
    NCCL_SYM(CommDestroy, "ncclCommDestroy")
    NCCL_SYM(AllGather, "ncclAllGather")
    NCCL_SYM(AllReduce, "ncclAllReduce")
    NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef NCCL_SYM
    return GANREV_OK;
}
#define NCCL_TRY(expr)                                                                                   \
    do {                                                                                                 \
        ncclResult_t r_ = (expr);                                                                        \
        if (r_ != ncclSuccess) return fail(ctx, GANREV_ENCCL, "%s failed: %s", #expr, ctx->nccl.GetErrorString(r_)); \
    } while (0)

int ganrev_comm_unique_id(ganrev_ctx* ctx, void* out, size_t cap, size_t* len) {
    if (!ctx || !out) return GANREV_EINVAL;
    if (cap < sizeof(ncclUniqueId)) return fail(ctx, GANREV_EINVAL, "unique id needs %zu bytes", sizeof(ncclUniqueId));
    RC_TRY(nccl_load(ctx));
    ncclUniqueId id;
    NCCL_TRY(ctx->nccl.GetUniqueId(&id));
    memcpy(out, &id, sizeof(id));
    if (len) *len = sizeof(id);
    return GANREV_OK;
}

int ganrev_comm_init(ganrev_ctx* ctx, int world, int rank, const void* uid, size_t len) {
    if (!ctx || !uid || world < 1 || rank < 0 || rank >= world) return ctx ? fail(ctx, GANREV_EINVAL, "bad comm arguments") : GANREV_EINVAL;
    if (len != sizeof(ncclUniqueId)) return fail(ctx, GANREV_EINVAL, "unique id must be %zu bytes", sizeof(ncclUniqueId));
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(nccl_load(ctx));
    ncclUniqueId id;
    memcpy(&id, uid, sizeof(id));
    NCCL_TRY(ctx->nccl.CommInitRank(&ctx->comm, world, id, rank));
    ctx->world = world; ctx->rank = rank;
    return GANREV_OK;
}

// ---------------------------------------------------------------- models
int ganrev_load_G(ganrev_ctx* ctx, int C, int H, int W, int noise_dim, const float* blob, size_t n_floats) {
    if (!ctx || !blob) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    return load_G_impl(ctx, C, H, W, noise_dim, blob, n_floats);
}
int ganrev_load_R(ganrev_ctx* ctx, int slot, int C, int H, int W, int noise_dim, int tanh_out, const float* blob, size_t n_floats) {
    if (!ctx || !blob) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    return load_R_impl(ctx, slot, C, H, W, noise_dim, tanh_out, blob, n_floats);
}

// ---------------------------------------------------------------- resident buffers
static size_t buf_row_bytes(ganrev_ctx* ctx, int which) {
    const int C = ctx->gC, H = ctx->gH, W = ctx->gW, nd = ctx->gnd;   // 0 until a model is loaded
    switch (which) {
        case GANREV_BUF_NOISE: case GANREV_BUF_ATTRS0: case GANREV_BUF_ATTRS1: return static_cast<size_t>(nd) * 4;
        case GANREV_BUF_IMAGES: case GANREV_BUF_FIXED: return static_cast<size_t>(C) * H * W * 4;
        case GANREV_BUF_MASK: return static_cast<size_t>(C) * H * W;
    }
    return 0;
}
// A resident buffer is about to be overwritten or reallocated: a database that aliases it is no longer set.
static void buf_touch(ganrev_ctx* ctx, int which) {
    if (which == GANREV_BUF_ATTRS0 && ctx->db_alias) { ctx->db_ptr = nullptr; ctx->db_alias = false; ctx->db_n = 0; ctx->assigned = false; }
}
static int buf_reserve(ganrev_ctx* ctx, int which, int64_t rows) {
    const size_t rb = buf_row_bytes(ctx, which);
    if (rb == 0) return fail(ctx, GANREV_ESTATE, "load a model before using resident buffers");
    buf_touch(ctx, which);
    RC_TRY(ensure(ctx, ctx->buf[which], rb * static_cast<size_t>(std::max<int64_t>(rows, 1))));
    return GANREV_OK;
}
int ganrev_buffer_put(ganrev_ctx* ctx, int which, const void* host, int64_t rows) {
    if (!ctx || !host || which < 0 || which >= GANREV_BUF_COUNT || rows < 0) return ctx ? fail(ctx, GANREV_EINVAL, "bad buffer_put arguments") : GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(buf_reserve(ctx, which, rows));
    CU_TRY(cudaMemcpyAsync(ctx->buf[which].p, host, buf_row_bytes(ctx, which) * rows, cudaMemcpyHostToDevice, ctx->stream));
    ctx->buf_rows[which] = rows;
    return finish(ctx);
}
int ganrev_buffer_get(ganrev_ctx* ctx, int which, void* host, int64_t row0, int64_t rows) {
    if (!ctx || !host || which < 0 || which >= GANREV_BUF_COUNT || rows < 0 || row0 < 0) return ctx ? fail(ctx, GANREV_EINVAL, "bad buffer_get arguments") : GANREV_EINVAL;
    if (row0 + rows > ctx->buf_rows[which]) return fail(ctx, GANREV_ESTATE, "buffer %d holds %lld rows", which, (long long)ctx->buf_rows[which]);
    CU_TRY(cudaSetDevice(ctx->device));
    const size_t rb = buf_row_bytes(ctx, which);
    CU_TRY(cudaMemcpyAsync(host, static_cast<const uint8_t*>(ctx->buf[which].p) + rb * row0, rb * rows, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

// input helper: host pointer -> upload into resident buffer; NULL -> resident buffer must hold >= N rows
static int stage_input(ganrev_ctx* ctx, int which, const void* host, int64_t N) {
    if (host) {
        RC_TRY(buf_reserve(ctx, which, N));   // (also un-sets a database aliasing this buffer)
        CU_TRY(cudaMemcpyAsync(ctx->buf[which].p, host, buf_row_bytes(ctx, which) * N, cudaMemcpyHostToDevice, ctx->stream));
        ctx->buf_rows[which] = N;
    } else if (ctx->buf_rows[which] < N || !ctx->buf[which].p) {
        return fail(ctx, GANREV_ESTATE, "resident buffer %d holds %lld rows, need %lld", which, (long long)ctx->buf_rows[which], (long long)N);
    }
    return GANREV_OK;
}
static int fetch_output(ganrev_ctx* ctx, int which, void* host, int64_t N) {
    if (host) CU_TRY(cudaMemcpyAsync(host, ctx->buf[which].p, buf_row_bytes(ctx, which) * N, cudaMemcpyDeviceToHost, ctx->stream));
    return GANREV_OK;
}

// ---------------------------------------------------------------- forward passes
int ganrev_forward_G(ganrev_ctx* ctx, const float* noise, int64_t N, float* images) {
    if (!ctx || N < 0) return ctx ? fail(ctx, GANREV_EINVAL, "bad forward_G arguments") : GANREV_EINVAL;
    if (!ctx->G.loaded) return fail(ctx, GANREV_ESTATE, "G not loaded");
    CU_TRY(cudaSetDevice(ctx->device));
    ChunkIO io;
    if (noise) {   // chunk-wise upload beside the kernels instead of one copy in front of them
        RC_TRY(buf_reserve(ctx, GANREV_BUF_NOISE, N));
        ctx->buf_rows[GANREV_BUF_NOISE] = N;
        io.h_in = reinterpret_cast<const uint8_t*>(noise); io.d_in = static_cast<uint8_t*>(ctx->buf[GANREV_BUF_NOISE].p); io.in_row = buf_row_bytes(ctx, GANREV_BUF_NOISE);
    } else {
        RC_TRY(stage_input(ctx, GANREV_BUF_NOISE, nullptr, N));
    }
    RC_TRY(buf_reserve(ctx, GANREV_BUF_IMAGES, N));
    if (images) { io.h_out = reinterpret_cast<uint8_t*>(images); io.d_out = static_cast<const uint8_t*>(ctx->buf[GANREV_BUF_IMAGES].p); io.out_row = buf_row_bytes(ctx, GANREV_BUF_IMAGES); }
    RC_TRY(forward_G_dev(ctx, static_cast<const float*>(ctx->buf[GANREV_BUF_NOISE].p), N, static_cast<float*>(ctx->buf[GANREV_BUF_IMAGES].p), &io));
    ctx->buf_rows[GANREV_BUF_IMAGES] = N;
    return finish(ctx);
}

int ganrev_forward_R(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N, float* attrs) {
    if (!ctx || N < 0 || slot < 0 || slot > 1) return ctx ? fail(ctx, GANREV_EINVAL, "bad forward_R arguments") : GANREV_EINVAL;
    if (!ctx->R[slot].loaded) return fail(ctx, GANREV_ESTATE, "R slot %d not loaded", slot);
    CU_TRY(cudaSetDevice(ctx->device));
    ChunkIO io;
    if (images) {
        RC_TRY(buf_reserve(ctx, GANREV_BUF_IMAGES, N));
        ctx->buf_rows[GANREV_BUF_IMAGES] = N;
        io.h_in = reinterpret_cast<const uint8_t*>(images); io.d_in = static_cast<uint8_t*>(ctx->buf[GANREV_BUF_IMAGES].p); io.in_row = buf_row_bytes(ctx, GANREV_BUF_IMAGES);
    } else {
        RC_TRY(stage_input(ctx, GANREV_BUF_IMAGES, nullptr, N));
    }
    const uint8_t* d_mask = nullptr;
    if (mask) {
        RC_TRY(stage_input(ctx, GANREV_BUF_MASK, mask, N));
        d_mask = static_cast<const uint8_t*>(ctx->buf[GANREV_BUF_MASK].p);
    }
    const int ob = slot == 0 ? GANREV_BUF_ATTRS0 : GANREV_BUF_ATTRS1;
    RC_TRY(buf_reserve(ctx, ob, N));
    if (attrs) { io.h_out = reinterpret_cast<uint8_t*>(attrs); io.d_out = static_cast<const uint8_t*>(ctx->buf[ob].p); io.out_row = buf_row_bytes(ctx, ob); }
    RC_TRY(forward_R_dev(ctx, slot, static_cast<const float*>(ctx->buf[GANREV_BUF_IMAGES].p), d_mask, N, static_cast<float*>(ctx->buf[ob].p), &io));
    ctx->buf_rows[ob] = N;
    return finish(ctx);
}

int ganrev_fix_l2(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N, float* attrs, float* fixed, double* l2) {
    if (!ctx || N < 0 || slot < 0 || slot > 1) return ctx ? fail(ctx, GANREV_EINVAL, "bad fix_l2 arguments") : GANREV_EINVAL;
    if (!ctx->R[slot].loaded || !ctx->G.loaded) return fail(ctx, GANREV_ESTATE, "fix_l2 needs G and R slot %d", slot);
    if (ctx->G.nd != ctx->R[slot].nd || ctx->G.C != ctx->R[slot].C || ctx->G.H != ctx->R[slot].H || ctx->G.W != ctx->R[slot].W)
        return fail(ctx, GANREV_ESTATE, "G and R geometries differ");
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(stage_input(ctx, GANREV_BUF_IMAGES, images, N));
    const uint8_t* d_mask = nullptr;
    if (mask) {
        RC_TRY(stage_input(ctx, GANREV_BUF_MASK, mask, N));
        d_mask = static_cast<const uint8_t*>(ctx->buf[GANREV_BUF_MASK].p);
    }
    const int ob = slot == 0 ? GANREV_BUF_ATTRS0 : GANREV_BUF_ATTRS1;
    RC_TRY(buf_reserve(ctx, ob, N));
    RC_TRY(buf_reserve(ctx, GANREV_BUF_FIXED, N));
    ctx->l2_valid = 0;
    RC_TRY(ensure(ctx, ctx->l2buf, sizeof(double) * static_cast<size_t>(std::max<int64_t>(N, 1))));
    const float* d_img = static_cast<const float*>(ctx->buf[GANREV_BUF_IMAGES].p);
    float* d_att = static_cast<float*>(ctx->buf[ob].p);
    float* d_fix = static_cast<float*>(ctx->buf[GANREV_BUF_FIXED].p);
    RC_TRY(forward_R_dev(ctx, slot, d_img, d_mask, N, d_att));
    ctx->buf_rows[ob] = N;
    RC_TRY(forward_G_dev(ctx, d_att, N, d_fix));
    ctx->buf_rows[GANREV_BUF_FIXED] = N;
    RC_TRY(l2_dev(ctx, d_img, d_fix, N, ctx->G.C * ctx->G.H * ctx->G.W, static_cast<double*>(ctx->l2buf.p)));
    ctx->l2_valid = N;
    RC_TRY(fetch_output(ctx, ob, attrs, N));
    RC_TRY(fetch_output(ctx, GANREV_BUF_FIXED, fixed, N));
    if (l2) CU_TRY(cudaMemcpyAsync(l2, ctx->l2buf.p, sizeof(double) * N, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

int ganrev_l2(ganrev_ctx* ctx, const float* a, const float* b, int64_t N, int px, double* l2) {
    if (!ctx || !a || !b || !l2 || N < 0 || px < 1) return ctx ? fail(ctx, GANREV_EINVAL, "bad l2 arguments") : GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    const size_t bytes = sizeof(float) * static_cast<size_t>(N) * px;
    RC_TRY(ensure(ctx, ctx->stage_a, bytes));
    RC_TRY(ensure(ctx, ctx->stage_b, bytes));
    ctx->l2_valid = 0;
    RC_TRY(ensure(ctx, ctx->l2buf, sizeof(double) * static_cast<size_t>(std::max<int64_t>(N, 1))));
    CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, a, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(ctx->stage_b.p, b, bytes, cudaMemcpyHostToDevice, ctx->stream));
    RC_TRY(l2_dev(ctx, static_cast<const float*>(ctx->stage_a.p), static_cast<const float*>(ctx->stage_b.p), N, px, static_cast<double*>(ctx->l2buf.p)));
    ctx->l2_valid = N;
    CU_TRY(cudaMemcpyAsync(l2, ctx->l2buf.p, sizeof(double) * N, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}


static int refine_check(ganrev_ctx* ctx) {
    if (!ctx->G.loaded) return fail(ctx, GANREV_ESTATE, "G not loaded");
    if (ctx->conv_impl != 0) return fail(ctx, GANREV_EINVAL, "refinement runs on the tcgen05 kernels only (conv_impl 0)");
    return GANREV_OK;
}

int ganrev_refine_l2(ganrev_ctx* ctx, int slot, const float* images, const float* z0, int64_t N, int iters, const float* hyper6,
                     float* attrs, float* fixed, double* l2) {
    if (!ctx || N < 0 || slot < 0 || slot > 1 || !hyper6) return ctx ? fail(ctx, GANREV_EINVAL, "bad refine_l2 arguments") : GANREV_EINVAL;
    if (iters < 0 || !(hyper6[0] > 0.0f) || !(hyper6[4] >= 0.0f))
        return fail(ctx, GANREV_EINVAL, "refine_l2 needs iters >= 0, lr > 0, prior >= 0 (got %d, %g, %g)", iters, hyper6[0], hyper6[4]);
    RC_TRY(refine_check(ctx));
    if (N == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(stage_input(ctx, GANREV_BUF_IMAGES, images, N));
    const int ob = slot == 0 ? GANREV_BUF_ATTRS0 : GANREV_BUF_ATTRS1;
    if (z0) {
        RC_TRY(stage_input(ctx, ob, z0, N));                  // (un-sets a database aliasing ATTRS0)
    } else {
        if (ctx->buf_rows[ob] < N || !ctx->buf[ob].p)
            return fail(ctx, GANREV_ESTATE, "resident buffer %d holds %lld rows, need %lld", ob, (long long)ctx->buf_rows[ob], (long long)N);
        buf_touch(ctx, ob);                                    // refined in place
    }
    RC_TRY(buf_reserve(ctx, GANREV_BUF_FIXED, N));
    ctx->l2_valid = 0;
    RC_TRY(ensure(ctx, ctx->l2buf, sizeof(double) * static_cast<size_t>(N)));
    const float* d_img = static_cast<const float*>(ctx->buf[GANREV_BUF_IMAGES].p);
    float* d_att = static_cast<float*>(ctx->buf[ob].p);
    float* d_fix = static_cast<float*>(ctx->buf[GANREV_BUF_FIXED].p);
    if (iters > 0) RC_TRY(refine_dev(ctx, d_img, d_att, N, iters, hyper6));
    // fixed / l2 from the same path as ganrev_fix_l2: bit-identical to ganrev_forward_G(z_final) + ganrev_l2
    RC_TRY(forward_G_dev(ctx, d_att, N, d_fix));
    ctx->buf_rows[GANREV_BUF_FIXED] = N;
    RC_TRY(l2_dev(ctx, d_img, d_fix, N, ctx->G.C * ctx->G.H * ctx->G.W, static_cast<double*>(ctx->l2buf.p)));
    ctx->l2_valid = N;
    RC_TRY(fetch_output(ctx, ob, attrs, N));
    RC_TRY(fetch_output(ctx, GANREV_BUF_FIXED, fixed, N));
    if (l2) CU_TRY(cudaMemcpyAsync(l2, ctx->l2buf.p, sizeof(double) * N, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

int ganrev_debug_refine_grad(ganrev_ctx* ctx, const float* images, const float* z, int64_t N, float prior, float* grad, double* f) {
    if (!ctx || !images || !z || !grad || !f || N < 0 || !(prior >= 0.0f)) return ctx ? fail(ctx, GANREV_EINVAL, "bad debug_refine_grad arguments") : GANREV_EINVAL;
    RC_TRY(refine_check(ctx));
    if (N == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    const GModel& G = ctx->G;
    GRefine& R = ctx->GR;
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, G.H, G.W), N);
    const long long px = static_cast<long long>(G.C) * G.H * G.W, nz = N * G.nd;
    RC_TRY(build_refine(ctx));
    RC_TRY(refine_buffers(ctx, CH));
    RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * N * px));
    RC_TRY(ensure(ctx, ctx->stage_b, sizeof(float) * nz));
    RC_TRY(ensure(ctx, R.zs, sizeof(float) * nz));
    RC_TRY(ensure(ctx, R.dist, sizeof(double) * N));
    const float* d_x = static_cast<const float*>(ctx->stage_a.p);
    const float* d_z = static_cast<const float*>(R.zs.p);
    float* d_g = static_cast<float*>(ctx->stage_b.p);
    double* d_dist = static_cast<double*>(R.dist.p);
    CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, images, sizeof(float) * N * px, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(R.zs.p, z, sizeof(float) * nz, cudaMemcpyHostToDevice, ctx->stream));
    for (int64_t n0 = 0; n0 < N; n0 += CH) {
        const int n = static_cast<int>(std::min<int64_t>(CH, N - n0));
        const long long ne = static_cast<long long>(n) * G.nd;
        RC_TRY(refine_grad_chunk(ctx, d_z + n0 * G.nd, d_x + n0 * px, n, CH));
        refine_grad_kernel<<<static_cast<unsigned>((ne + 255) / 256), 256, 0, ctx->stream>>>(static_cast<const float*>(R.glin.p), d_z + n0 * G.nd, 2.0f * prior, d_g + n0 * G.nd, ne);
        CU_TRY(cudaGetLastError());
        RC_TRY(l2_dev(ctx, d_x + n0 * px, static_cast<const float*>(R.y.p), n, static_cast<int>(px), d_dist + n0));
    }
    std::vector<double> dist(N);
    CU_TRY(cudaMemcpyAsync(grad, d_g, sizeof(float) * nz, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaMemcpyAsync(dist.data(), d_dist, sizeof(double) * N, cudaMemcpyDeviceToHost, ctx->stream));
    RC_TRY(finish(ctx));
    for (int64_t i = 0; i < N; ++i) {   // f = ||G(z) - x||^2 + prior ||z||^2
        double zz = 0.0;
        for (int k = 0; k < G.nd; ++k) zz += static_cast<double>(z[i * G.nd + k]) * z[i * G.nd + k];
        f[i] = dist[i] * dist[i] + static_cast<double>(prior) * zz;
    }
    return GANREV_OK;
}

int ganrev_debug_refine_stage(ganrev_ctx* ctx, const float* images, const float* z, int64_t N, int stage, void* out, size_t out_bytes) {
    if (!ctx || !images || !z || !out || N < 0 || stage < 0 || stage >= RSTAGE_COUNT)
        return ctx ? fail(ctx, GANREV_EINVAL, "bad debug_refine_stage arguments (stage %d)", stage) : GANREV_EINVAL;
    RC_TRY(refine_check(ctx));
    const GModel& G = ctx->G;
    GRefine& R = ctx->GR;
    const size_t px = static_cast<size_t>(G.H) * G.W;
    const size_t row[RSTAGE_COUNT] = {static_cast<size_t>(G.F) * 2, px / 4 * 256 * 2, px * 128 * 2, static_cast<size_t>(G.C) * px * 4,
                                      px * 128 * 2, px / 4 * 256 * 2, static_cast<size_t>(G.F) * 2, static_cast<size_t>(G.nd) * 4};
    if (out_bytes != row[stage] * static_cast<size_t>(N))
        return fail(ctx, GANREV_EINVAL, "debug_refine_stage: out_bytes %zu, stage %d of %lld rows needs %zu", out_bytes, stage, (long long)N, row[stage] * static_cast<size_t>(N));
    if (N == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, G.H, G.W), N);
    const long long pxc = static_cast<long long>(G.C) * px, nz = N * G.nd;
    RC_TRY(build_refine(ctx));
    RC_TRY(refine_buffers(ctx, CH));
    RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * N * pxc));
    RC_TRY(ensure(ctx, R.zs, sizeof(float) * nz));
    const float* d_x = static_cast<const float*>(ctx->stage_a.p);
    const float* d_z = static_cast<const float*>(R.zs.p);
    CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, images, sizeof(float) * N * pxc, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(R.zs.p, z, sizeof(float) * nz, cudaMemcpyHostToDevice, ctx->stream));
    const void* src[RSTAGE_COUNT] = {R.h0.p, R.h1.p, R.h2.p, R.y.p, ctx->arena[0].p, ctx->arena[1].p, ctx->arena[0].p, R.glin.p};
    for (int64_t n0 = 0; n0 < N; n0 += CH) {   // chunks as ganrev_debug_refine_grad runs them; rows land in input order
        const int n = static_cast<int>(std::min<int64_t>(CH, N - n0));
        RC_TRY(refine_grad_chunk(ctx, d_z + n0 * G.nd, d_x + n0 * pxc, n, CH, stage));
        CU_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(out) + n0 * row[stage], src[stage], row[stage] * n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return finish(ctx);
}

// Forward layer hooks: forward_G_dev / forward_R_dev run one chunk at a time (n <= the chunk size forward_G / forward_R use, so every
// layer sees the shapes it sees there), stopped after `stage`; that layer's buffer is copied out after each chunk, rows in input order.
int ganrev_debug_G_stage(ganrev_ctx* ctx, const float* noise, int64_t N, int stage, void* out, size_t out_bytes) {
    if (!ctx || !noise || !out || N < 0 || stage < 0 || stage >= GLAYER_COUNT)
        return ctx ? fail(ctx, GANREV_EINVAL, "bad debug_G_stage arguments (stage %d)", stage) : GANREV_EINVAL;
    GModel& G = ctx->G;
    if (!G.loaded) return fail(ctx, GANREV_ESTATE, "G not loaded");
    const bool fused = G.fuse3 && ctx->conv_impl == 0;
    if (stage == GLAYER_C2 && fused) return fail(ctx, GANREV_ESTATE, "debug_G_stage: conv2's activation is never stored when the tap products are fused");
    const size_t px = static_cast<size_t>(G.H) * G.W;
    const size_t row[GLAYER_COUNT] = {static_cast<size_t>(G.F) * 2, px / 4 * 256 * 2, px * 128 * 2, 9 * static_cast<size_t>(G.C) * px * 4,
                                      static_cast<size_t>(G.C) * px * 4};
    if (out_bytes != row[stage] * static_cast<size_t>(N))
        return fail(ctx, GANREV_EINVAL, "debug_G_stage: out_bytes %zu, stage %d of %lld rows needs %zu", out_bytes, stage, (long long)N, row[stage] * static_cast<size_t>(N));
    if (N == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, G.H, G.W), N);
    RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * N * G.nd));
    RC_TRY(ensure(ctx, ctx->stage_b, sizeof(float) * CH * G.C * px));
    CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, noise, sizeof(float) * N * G.nd, cudaMemcpyHostToDevice, ctx->stream));
    const float* d_noise = static_cast<const float*>(ctx->stage_a.p);
    float* d_img = static_cast<float*>(ctx->stage_b.p);
    uint8_t* o = static_cast<uint8_t*>(out);
    for (int64_t n0 = 0; n0 < N; n0 += CH) {
        const int64_t n = std::min<int64_t>(CH, N - n0);
        RC_TRY(forward_G_dev(ctx, d_noise + n0 * G.nd, n, d_img, nullptr, stage));
        if (stage == GLAYER_TAPS) {   // plane k of P[k][pixel] (stride: forward_G_dev's chunk of n images) -> out[image][k][H][W]
            const float* planes = static_cast<const float*>(ctx->arena[fused ? 0 : 1].p);
            for (int k = 0; k < 9 * G.C; ++k)
                CU_TRY(cudaMemcpy2DAsync(o + n0 * row[stage] + k * px * 4, row[stage], planes + k * n * px, px * 4, px * 4, n,
                                         cudaMemcpyDeviceToHost, ctx->stream));
        } else {
            const void* src[GLAYER_COUNT] = {ctx->arena[0].p, ctx->arena[1].p, ctx->arena[0].p, nullptr, d_img};
            CU_TRY(cudaMemcpyAsync(o + n0 * row[stage], src[stage], row[stage] * n, cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    return finish(ctx);
}

int ganrev_debug_R_stage(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N, int stage, void* out, size_t out_bytes) {
    if (!ctx || !images || !out || N < 0 || slot < 0 || slot > 1 || stage < 0 || stage >= RLAYER_COUNT)
        return ctx ? fail(ctx, GANREV_EINVAL, "bad debug_R_stage arguments (slot %d, stage %d)", slot, stage) : GANREV_EINVAL;
    RModel& R = ctx->R[slot];
    if (!R.loaded) return fail(ctx, GANREV_ESTATE, "R slot %d not loaded", slot);
    const size_t px = static_cast<size_t>(R.H) * R.W, pxc = static_cast<size_t>(R.C) * px;
    const size_t row[RLAYER_COUNT] = {px * 64 * 2, px * 64 * 2, px / 4 * 64 * 2, px / 4 * 128 * 2, px / 4 * 128 * 2, px / 16 * 128 * 2,
                                      512 * 2, static_cast<size_t>(R.nd) * 4};
    if (out_bytes != row[stage] * static_cast<size_t>(N))
        return fail(ctx, GANREV_EINVAL, "debug_R_stage: out_bytes %zu, stage %d of %lld rows needs %zu", out_bytes, stage, (long long)N, row[stage] * static_cast<size_t>(N));
    if (N == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    const int64_t CH = std::min<int64_t>(chunk_for(ctx, R.H, R.W), N);
    // stage_a: the images; stage_b: the output vectors of one chunk, then the dropout mask
    const size_t attr_bytes = sizeof(float) * CH * R.nd;
    RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * N * pxc));
    RC_TRY(ensure(ctx, ctx->stage_b, attr_bytes + (mask ? N * pxc : 0)));
    CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, images, sizeof(float) * N * pxc, cudaMemcpyHostToDevice, ctx->stream));
    const uint8_t* d_mask = nullptr;
    if (mask) {
        d_mask = static_cast<const uint8_t*>(ctx->stage_b.p) + attr_bytes;
        CU_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(ctx->stage_b.p) + attr_bytes, mask, N * pxc, cudaMemcpyHostToDevice, ctx->stream));
    }
    const float* d_img = static_cast<const float*>(ctx->stage_a.p);
    float* d_att = static_cast<float*>(ctx->stage_b.p);
    for (int64_t n0 = 0; n0 < N; n0 += CH) {
        const int64_t n = std::min<int64_t>(CH, N - n0);
        RC_TRY(forward_R_dev(ctx, slot, d_img + n0 * pxc, d_mask ? d_mask + n0 * pxc : nullptr, n, d_att, nullptr, stage));
        // the layers alternate between the two arenas, conv1 writing arena[0]
        const void* s = stage == RLAYER_OUT ? static_cast<const void*>(d_att) : ctx->arena[stage & 1].p;
        CU_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(out) + n0 * row[stage], s, row[stage] * n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return finish(ctx);
}

}  // extern "C"
static int tfs_make_map(ganrev_ctx* ctx, CUtensorMap* m, const float* base, int d, long long rows);
extern "C" {
int ganrev_nearest_l2(ganrev_ctx* ctx, const float* queries, int Q, const float* set, int64_t N, int px, int64_t* ids, double* dist) {
    if (!ctx || !queries || Q < 0 || N < 0 || px < 1 || !ids || !dist) return ctx ? fail(ctx, GANREV_EINVAL, "bad nearest_l2 arguments") : GANREV_EINVAL;
    if (Q == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    const float* d_set = nullptr;
    if (set) {
        RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * static_cast<size_t>(std::max<int64_t>(N, 1)) * px));
        if (N > 0) CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, set, sizeof(float) * static_cast<size_t>(N) * px, cudaMemcpyHostToDevice, ctx->stream));
        d_set = static_cast<const float*>(ctx->stage_a.p);
    } else {
        if (ctx->buf_rows[GANREV_BUF_IMAGES] < N || (N > 0 && buf_row_bytes(ctx, GANREV_BUF_IMAGES) != sizeof(float) * static_cast<size_t>(px)))
            return fail(ctx, GANREV_ESTATE, "resident IMAGES do not hold %lld rows of %d floats", (long long)N, px);
        d_set = static_cast<const float*>(ctx->buf[GANREV_BUF_IMAGES].p);
    }
    RC_TRY(ensure(ctx, ctx->stage_b, sizeof(float) * static_cast<size_t>(Q) * px));
    CU_TRY(cudaMemcpyAsync(ctx->stage_b.p, queries, sizeof(float) * static_cast<size_t>(Q) * px, cudaMemcpyHostToDevice, ctx->stream));
    // one warp per set row, 8 warps per block, a few blocks per SM; never more warps than rows
    const long long want_warps = std::max<long long>(1, std::min<long long>(N, 8LL * 4 * ctx->num_sms));
    const int blocks = static_cast<int>((want_warps + 7) / 8);
    const long long n_warps = 8LL * blocks;
    RC_TRY(ensure(ctx, ctx->nn_partial, sizeof(NearestRec) * static_cast<size_t>(n_warps) * NL2_QB));
    RC_TRY(ensure(ctx, ctx->nn_ids, sizeof(long long) * static_cast<size_t>(Q)));
    RC_TRY(ensure(ctx, ctx->nn_dist, sizeof(double) * static_cast<size_t>(Q)));
    RC_TRY(ensure(ctx, ctx->nn_flag, static_cast<size_t>(Q)));
    CU_TRY(cudaMemsetAsync(ctx->nn_flag.p, 0, static_cast<size_t>(Q), ctx->stream));
    // tensor-core filter + canonical evaluation of the candidates (nearest_tc.cuh) where the shape allows, else the exact kernel for every pair
    const int tc_nbox = (px + tfs::kBoxCols - 1) / tfs::kBoxCols;
    const size_t tc_fixed = ntc::nearest_fixed_bytes(px) + 1024;
    const bool use_tc = ctx->stream_tc && N >= 1 && N <= 0x7fffff00LL && px % 4 == 0 && (reinterpret_cast<uintptr_t>(d_set) & 15) == 0 &&
                        tc_fixed + 4 * static_cast<size_t>(tfs::kSlotBytes) <= 227 * 1024;
    if (use_tc) {
        const int nslots = static_cast<int>(std::min<size_t>(tfs::kMaxSlots, (227 * 1024 - tc_fixed) / tfs::kSlotBytes));
        const size_t smem = tc_fixed + static_cast<size_t>(nslots) * tfs::kSlotBytes;
        const long long n_tiles = (N + tfs::kRows - 1) / tfs::kRows;
        const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(n_tiles, ctx->num_sms)));
        const long long tc_warps = 4LL * grid;
        RC_TRY(ensure(ctx, ctx->nn_partial, sizeof(NearestRec) * static_cast<size_t>(std::max(n_warps, tc_warps)) * NL2_QB));
        if (!ctx->tfs_aux.p) {
            RC_TRY(ensure(ctx, ctx->tfs_aux, 32 * sizeof(unsigned) + 4 * sizeof(unsigned long long)));
            CU_TRY(cudaMemsetAsync(ctx->tfs_aux.p, 0, 32 * sizeof(unsigned) + 4 * sizeof(unsigned long long), ctx->stream));
        }
        static size_t attr_max_dev[kMaxDevices] = {};
        size_t& attr_max = attr_max_dev[ctx->device];
        if (smem > attr_max) {
            CU_TRY(cudaFuncSetAttribute(ntc::nearest_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            attr_max = smem;
        }
        CUtensorMap tm;
        RC_TRY(tfs_make_map(ctx, &tm, d_set, px, N));
        for (int q0 = 0; q0 < Q; q0 += NL2_QB) {
            const int nq = std::min(NL2_QB, Q - q0);
            ntc::NParams np{};
            np.set = d_set; np.n_rows = N; np.px = px; np.q = static_cast<const float*>(ctx->stage_b.p); np.q0 = q0; np.nq = nq;
            np.partial = static_cast<NearestRec*>(ctx->nn_partial.p); np.row0_nan = static_cast<unsigned char*>(ctx->nn_flag.p);
            np.gthr = static_cast<unsigned*>(ctx->tfs_aux.p);
            np.stats = reinterpret_cast<unsigned long long*>(np.gthr + 32);
            np.n_tiles = n_tiles; np.nbox = tc_nbox; np.nslots = nslots; np.err_flag = ctx->d_err_flag;
            {
                ProfScope ps(ctx, "nearest_l2", 3.0 * N * px * nq, 4.0 * N * px);
                ntc::nearest_init_kernel<<<1, 32, 0, ctx->stream>>>(np.gthr);
                ntc::nearest_tc_kernel<<<grid, ntc::kThreads, smem, ctx->stream>>>(tm, np);
                ctx->launches++;
                ctx->tfs_launches++;
                CU_TRY(cudaGetLastError());
            }
            {
                ProfScope ps(ctx, "nearest_l2_merge", 0.0, 16.0 * tc_warps * nq);
                nearest_l2_merge_kernel<<<nq, 32, 0, ctx->stream>>>(static_cast<const NearestRec*>(ctx->nn_partial.p), tc_warps, Q, q0, N,
                                                                   static_cast<const unsigned char*>(ctx->nn_flag.p), ctx->world == 1 ? 1 : 0,
                                                                   static_cast<long long*>(ctx->nn_ids.p), static_cast<double*>(ctx->nn_dist.p));
                CU_TRY(cudaGetLastError());
            }
        }
    }
    for (int q0 = 0; q0 < Q && !use_tc; q0 += NL2_QB) {
        const int nq = std::min(NL2_QB, Q - q0);
        {
            ProfScope ps(ctx, "nearest_l2", 3.0 * N * px * nq, 4.0 * N * px);
            nearest_l2_kernel<<<blocks, 256, 0, ctx->stream>>>(static_cast<const float*>(ctx->stage_b.p), Q, q0, d_set, N, px,
                                                               static_cast<NearestRec*>(ctx->nn_partial.p), static_cast<unsigned char*>(ctx->nn_flag.p));
            CU_TRY(cudaGetLastError());
        }
        {
            ProfScope ps(ctx, "nearest_l2_merge", 0.0, 16.0 * n_warps * nq);
            nearest_l2_merge_kernel<<<nq, 32, 0, ctx->stream>>>(static_cast<const NearestRec*>(ctx->nn_partial.p), n_warps, Q, q0, N,
                                                               static_cast<const unsigned char*>(ctx->nn_flag.p), ctx->world == 1 ? 1 : 0,
                                                               static_cast<long long*>(ctx->nn_ids.p), static_cast<double*>(ctx->nn_dist.p));
            CU_TRY(cudaGetLastError());
        }
    }
    if (ctx->world > 1) {
        // row-sharded set (each rank passes its own shard): global row = local row + the lower ranks' N; one allgather of
        // Q records, merged identically on every rank; the "row 0 sticks" quirk belongs to the rank that owns global row 0
        RC_TRY(ensure(ctx, ctx->shard, sizeof(long long) * (ctx->world + 2)));
        long long* d_all = static_cast<long long*>(ctx->shard.p);
        const long long mine = N;
        std::vector<long long> all(ctx->world, 0);
        CU_TRY(cudaMemcpyAsync(d_all + ctx->world, &mine, sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        NCCL_TRY(ctx->nccl.AllGather(d_all + ctx->world, d_all, 1, ncclInt64, ctx->comm, ctx->stream));
        CU_TRY(cudaMemcpyAsync(all.data(), d_all, sizeof(long long) * ctx->world, cudaMemcpyDeviceToHost, ctx->stream));
        RC_TRY(finish(ctx));
        long long offset = 0, total = 0;
        for (int r = 0; r < ctx->world; ++r) { if (r < ctx->rank) offset += all[r]; total += all[r]; }
        RC_TRY(ensure(ctx, ctx->nn_all, sizeof(NearestRankRec) * static_cast<size_t>(Q) * (ctx->world + 1)));
        NearestRankRec* rec_all = static_cast<NearestRankRec*>(ctx->nn_all.p);
        NearestRankRec* rec_mine = rec_all + static_cast<size_t>(Q) * ctx->world;
        ProfScope ps(ctx, "nearest_l2_ranks", 0.0, 32.0 * Q * ctx->world);
        nearest_l2_pack_kernel<<<(Q + 127) / 128, 128, 0, ctx->stream>>>(static_cast<const long long*>(ctx->nn_ids.p), static_cast<const double*>(ctx->nn_dist.p),
            static_cast<const unsigned char*>(ctx->nn_flag.p), Q, offset, (offset == 0 && N > 0) ? 1 : 0, rec_mine);
        NCCL_TRY(ctx->nccl.AllGather(rec_mine, rec_all, sizeof(NearestRankRec) * static_cast<size_t>(Q), ncclUint8, ctx->comm, ctx->stream));
        nearest_l2_ranks_kernel<<<(Q + 127) / 128, 128, 0, ctx->stream>>>(rec_all, ctx->world, Q, total, static_cast<long long*>(ctx->nn_ids.p), static_cast<double*>(ctx->nn_dist.p));
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "ids are copied out as int64");
    CU_TRY(cudaMemcpyAsync(ids, ctx->nn_ids.p, sizeof(int64_t) * Q, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaMemcpyAsync(dist, ctx->nn_dist.p, sizeof(double) * Q, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

int ganrev_anomaly_flags(ganrev_ctx* ctx, const double* l2, int64_t n_calc, int64_t n_show, double quantile, uint8_t* flags, double* thr) {
    if (!ctx || n_calc < 0 || n_show < 0 || n_show > n_calc || (!flags && n_show > 0)) return ctx ? fail(ctx, GANREV_EINVAL, "bad anomaly_flags arguments") : GANREV_EINVAL;
    if (ctx->world == 1 && n_calc < 1) return fail(ctx, GANREV_EINVAL, "bad anomaly_flags arguments");
    if (!l2 && ctx->l2_valid < n_calc) return fail(ctx, GANREV_ESTATE, "l2 == NULL needs %lld resident distances, the last fix_l2 / l2 call left %lld", (long long)n_calc, (long long)ctx->l2_valid);
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(ensure(ctx, ctx->qsel, sizeof(unsigned long long) * (4 + 256)));
    unsigned long long* state = static_cast<unsigned long long*>(ctx->qsel.p);
    unsigned long long* hist = state + 4;
    int64_t n_total = n_calc;
    if (ctx->world > 1) {   // the distances are sharded like the images: the order statistic is over all ranks' n_calc values
        const unsigned long long mine = static_cast<unsigned long long>(n_calc);
        CU_TRY(cudaMemcpyAsync(state + 2, &mine, sizeof(mine), cudaMemcpyHostToDevice, ctx->stream));
        NCCL_TRY(ctx->nccl.AllReduce(state + 2, state + 2, 1, ncclUint64, ncclSum, ctx->comm, ctx->stream));
        unsigned long long tot = 0;
        CU_TRY(cudaMemcpyAsync(&tot, state + 2, sizeof(tot), cudaMemcpyDeviceToHost, ctx->stream));
        RC_TRY(finish(ctx));
        n_total = static_cast<int64_t>(tot);
    }
    const int64_t r = static_cast<int64_t>(std::floor(static_cast<double>(n_total) * quantile));   // math.floor(#distancesForSort*threshold)
    if (r < 1 || r > n_total) return fail(ctx, GANREV_EINVAL, "floor(n_calc*quantile)=%lld is not a valid 1-based index", (long long)r);
    if (l2 || n_calc == 0) RC_TRY(ensure(ctx, ctx->l2buf, sizeof(double) * static_cast<size_t>(std::max<int64_t>(n_calc, 1))));
    RC_TRY(ensure(ctx, ctx->thr, sizeof(double)));
    RC_TRY(ensure(ctx, ctx->flags, static_cast<size_t>(std::max<int64_t>(n_show, 1))));
    if (l2 && n_calc > 0) { CU_TRY(cudaMemcpyAsync(ctx->l2buf.p, l2, sizeof(double) * n_calc, cudaMemcpyHostToDevice, ctx->stream)); ctx->l2_valid = n_calc; }
    {
        ProfScope ps(ctx, "quantile_select", 0.0, 8.0 * 8.0 * n_calc);
        ctx->launches += 16;
        quantile_init_kernel<<<1, 256, 0, ctx->stream>>>(state, hist, r - 1, quantile);
        const int blocks = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n_calc + 4095) / 4096, 4LL * ctx->num_sms)));
        for (int pass = 0; pass < 8; ++pass) {
            quantile_hist_kernel<<<blocks, 256, 0, ctx->stream>>>(static_cast<const double*>(ctx->l2buf.p), n_calc, state, pass, hist);
            if (ctx->world > 1) NCCL_TRY(ctx->nccl.AllReduce(hist, hist, 256, ncclUint64, ncclSum, ctx->comm, ctx->stream));
            quantile_pick_kernel<<<1, 256, 0, ctx->stream>>>(state, hist, pass, static_cast<double*>(ctx->thr.p));
        }
        CU_TRY(cudaGetLastError());
    }
    if (n_show > 0) {
        ProfScope ps(ctx, "anomaly_flags", 0.0, 9.0 * n_show);
        anomaly_flags_kernel<<<static_cast<unsigned>((n_show + 255) / 256), 256, 0, ctx->stream>>>(
            static_cast<const double*>(ctx->l2buf.p), n_show, static_cast<const double*>(ctx->thr.p), static_cast<uint8_t*>(ctx->flags.p));
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaMemcpyAsync(flags, ctx->flags.p, n_show, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (thr) CU_TRY(cudaMemcpyAsync(thr, ctx->thr.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

// ---------------------------------------------------------------- database
static int vec_prep(ganrev_ctx* ctx, const float* x, int64_t n, int d, float* rn, float* halfsq, unsigned int* maxabs) {
    ProfScope ps(ctx, "vec_prep", 2.0 * n * d, 4.0 * n * d);
    if (n > 0) scan::vec_prep_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, ctx->stream>>>(x, n, d, rn, halfsq, maxabs);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

static int db_set_impl(ganrev_ctx* ctx, const float* vecs, int64_t N, int d, bool own_resident);
int ganrev_db_set(ganrev_ctx* ctx, const float* vecs, int64_t N, int d) { return db_set_impl(ctx, vecs, N, d, false); }
static int ganrev_db_adopt_own(ganrev_ctx* ctx, int64_t N, int d) { return db_set_impl(ctx, nullptr, N, d, true); }
// own_resident: ctx->db already holds the rows on the device (ganrev_debug_db_synthetic)
static int db_set_impl(ganrev_ctx* ctx, const float* vecs, int64_t N, int d, bool own_resident) {
    if (!ctx || N < 0 || d < 1 || N > 0xFFFFFFF0ll) return ctx ? fail(ctx, GANREV_EINVAL, "bad db_set arguments") : GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    const size_t bytes = sizeof(float) * static_cast<size_t>(N) * d;
    ctx->db_ptr = nullptr; ctx->db_alias = false; ctx->db_n = 0; ctx->assigned = false; ctx->pdb_valid = false;
    RC_TRY(ensure(ctx, ctx->rdb, sizeof(float) * static_cast<size_t>(std::max<int64_t>(N, 1))));
    RC_TRY(ensure(ctx, ctx->maxabs, 3 * sizeof(long long)));
    RC_TRY(ensure(ctx, ctx->shard, sizeof(long long) * (ctx->world + 2)));
    const float* rows = nullptr;
    if (own_resident) {
        rows = static_cast<const float*>(ctx->db.p);
    } else if (vecs) {
        RC_TRY(ensure(ctx, ctx->db, bytes));
        CU_TRY(cudaMemcpyAsync(ctx->db.p, vecs, bytes, cudaMemcpyHostToDevice, ctx->stream));
        rows = static_cast<const float*>(ctx->db.p);
    } else {
        // the recovered vectors stay where R left them: the database ALIASES the resident ATTRS0 buffer (no copy);
        // overwriting ATTRS0 afterwards (forward_R / fix_l2 slot 0, buffer_put) un-sets the database
        if (ctx->buf_rows[GANREV_BUF_ATTRS0] < N || !ctx->buf[GANREV_BUF_ATTRS0].p || buf_row_bytes(ctx, GANREV_BUF_ATTRS0) != sizeof(float) * static_cast<size_t>(d))
            return fail(ctx, GANREV_ESTATE, "resident ATTRS0 does not hold %lld x %d", (long long)N, d);
        rows = static_cast<const float*>(ctx->buf[GANREV_BUF_ATTRS0].p);
    }
    CU_TRY(cudaMemsetAsync(ctx->maxabs.p, 0, 3 * sizeof(long long), ctx->stream));
    RC_TRY(vec_prep(ctx, rows, N, d, static_cast<float*>(ctx->rdb.p), nullptr, static_cast<unsigned int*>(ctx->maxabs.p)));
    unsigned int mb = 0;
    std::vector<long long> all(ctx->world, 0);
    if (ctx->world > 1) {
        // row-shard bookkeeping: global offset = sum of the lower ranks' N; global max|x| (one allgather + one allreduce, no allocation)
        long long* d_all = static_cast<long long*>(ctx->shard.p);
        const long long mine = N;
        CU_TRY(cudaMemcpyAsync(d_all + ctx->world, &mine, sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        {
            ProfScope pc(ctx, "nccl_shard_bookkeeping", 0.0, 12.0 * ctx->world, false);
            NCCL_TRY(ctx->nccl.AllGather(d_all + ctx->world, d_all, 1, ncclInt64, ctx->comm, ctx->stream));
            NCCL_TRY(ctx->nccl.AllReduce(ctx->maxabs.p, ctx->maxabs.p, 1, ncclUint32, ncclMax, ctx->comm, ctx->stream));
        }
        CU_TRY(cudaMemcpyAsync(all.data(), d_all, sizeof(long long) * ctx->world, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU_TRY(cudaMemcpyAsync(&mb, ctx->maxabs.p, sizeof(mb), cudaMemcpyDeviceToHost, ctx->stream));
    RC_TRY(finish(ctx));
    memcpy(&ctx->db_maxabs, &mb, 4);
    ctx->db_offset = 0; ctx->db_total = N;
    if (ctx->world > 1) {
        ctx->db_total = 0;
        for (int r = 0; r < ctx->world; ++r) { if (r < ctx->rank) ctx->db_offset += all[r]; ctx->db_total += all[r]; }
        if (ctx->db_total > 0xFFFFFFF0ll) return fail(ctx, GANREV_EINVAL, "global database exceeds 2^32 rows");
    }
    ctx->db_ptr = rows; ctx->db_alias = vecs == nullptr && !own_resident; ctx->db_n = N; ctx->db_d = d;
    return GANREV_OK;
}

int ganrev_cosine(ganrev_ctx* ctx, const float* a, const float* b, int d, float* out) {
    if (!ctx || !a || !b || !out || d < 1) return ctx ? fail(ctx, GANREV_EINVAL, "bad cosine arguments") : GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * (2 * static_cast<size_t>(d) + 1)));
    float* da = static_cast<float*>(ctx->stage_a.p);
    CU_TRY(cudaMemcpyAsync(da, a, sizeof(float) * d, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(da + d, b, sizeof(float) * d, cudaMemcpyHostToDevice, ctx->stream));
    {
        ProfScope ps(ctx, "cosine_pair", 6.0 * d, 8.0 * d);
        scan::cosine_pair_kernel<<<1, 32, 0, ctx->stream>>>(da, da + d, d, da + 2 * d);
        CU_TRY(cudaGetLastError());
    }
    CU_TRY(cudaMemcpyAsync(out, da + 2 * d, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

}  // extern "C"
template <int TQ, int E>
static int launch_search(ganrev_ctx* ctx, const scan::ScanParams& p, int splits) {
    constexpr int QT = 16 * TQ, K2 = 32 * E;
    const size_t smem = sizeof(float) * (scan::DK * scan::XS + scan::DK * QT) + sizeof(unsigned long long) * (QT * K2 + QT * scan::CAP + QT) + sizeof(int) * QT;
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(scan::search_kernel<TQ, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    dim3 grid(splits, (p.nq + QT - 1) / QT);
    scan::search_kernel<TQ, E><<<grid, scan::kThreads, smem, ctx->stream>>>(p);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

extern "C" {
}  // extern "C"
template <int E>
static int launch_search_wide(ganrev_ctx* ctx, const scan::ScanParams& p, int splits) {
    constexpr int QT = 64, K2 = 32 * E;
    const size_t smem = sizeof(float) * (static_cast<size_t>(p.d) * scan::XS + static_cast<size_t>(p.d) * QT) +
                        sizeof(unsigned long long) * (QT * K2 + QT * scan::CAP + QT) + sizeof(int) * QT;
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(scan::search_kernel_wide<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    dim3 grid(splits, (p.nq + QT - 1) / QT);
    scan::search_kernel_wide<E><<<grid, scan::kThreads, smem, ctx->stream>>>(p);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

template <int E>
static int launch_search_wide4(ganrev_ctx* ctx, const scan::ScanParams& p, int splits) {
    constexpr int QT = 64, K2 = 32 * E;
    const int S = scan::wide4_stride(p.d);
    const size_t smem = sizeof(float) * (static_cast<size_t>(scan::RT + QT) * S) +
                        sizeof(unsigned long long) * (QT * K2 + QT * scan::CAP + QT) + sizeof(int) * QT;
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(scan::search_kernel_wide4<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    dim3 grid(splits, (p.nq + QT - 1) / QT);
    scan::search_kernel_wide4<E><<<grid, scan::kThreads, smem, ctx->stream>>>(p);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

// ---- streaming kernels (nq <= 32, d % 4 == 0): plan + launch
static bool stream_plan(ganrev_ctx* ctx, const scan::ScanParams& p, int NQ, int mode, int K2, scan::StreamParams& sp, size_t& smem, int& grid) {
    if (p.d % 4 != 0 || p.nq > 32) return false;
    if (mode == 1 && p.d > 128) return false;                 // the update pass needs the whole row tile in smem
    sp.s = p;
    sp.dc = std::min(p.d, 128);
    sp.dc_pad = sp.dc + (((sp.dc / 4) % 2 == 0) ? 4 : 0);     // odd number of 16-byte pieces per row: conflict-free
    sp.n_chunks = (p.d + sp.dc - 1) / sp.dc;
    sp.c4_magic = static_cast<unsigned>(((1ull << 32) + (sp.dc / 4) - 1) / (sp.dc / 4));
    sp.groups = mode == 1 ? std::max(1, scan::kThreads / (p.d / 4)) : 0;      // thread groups of d/4 threads (4 columns each)
    smem = sizeof(float) * (static_cast<size_t>(scan::SSTAGES) * scan::SR * sp.dc_pad + static_cast<size_t>(p.d) * NQ);
    if (mode == 0) smem += sizeof(unsigned long long) * (static_cast<size_t>(NQ) * K2 + NQ * scan::CAP + NQ) + sizeof(int) * NQ;
    else smem += (mode == 1 ? sizeof(unsigned long long) * (static_cast<size_t>(p.nq) * p.d + p.nq) : 0) + 4 * sizeof(int) * scan::SR;
    if (smem > 220 * 1024) return false;
    const long long n_tiles = (p.n_rows + scan::SR - 1) / scan::SR;
    grid = static_cast<int>(std::max<long long>(1, std::min<long long>(n_tiles, ctx->num_sms)));
    sp.tiles_per_block = (n_tiles + grid - 1) / grid;
    grid = static_cast<int>(std::max<long long>(1, (n_tiles + sp.tiles_per_block - 1) / sp.tiles_per_block));
    return true;
}
template <int NQ, int MODE, int E>
static int launch_stream(ganrev_ctx* ctx, const scan::StreamParams& sp, size_t smem, int grid) {
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(scan::stream_kernel<NQ, MODE, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    scan::stream_kernel<NQ, MODE, E><<<grid, scan::kThreads, smem, ctx->stream>>>(sp);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}
template <int MODE, int E>
static int dispatch_stream(ganrev_ctx* ctx, int NQ, const scan::StreamParams& sp, size_t smem, int grid) {
    switch (NQ) {
        case 4: return launch_stream<4, MODE, E>(ctx, sp, smem, grid);
        case 8: return launch_stream<8, MODE, E>(ctx, sp, smem, grid);
        case 16: return launch_stream<16, MODE, E>(ctx, sp, smem, grid);
        case 24: return launch_stream<24, MODE, E>(ctx, sp, smem, grid);
        case 32: return launch_stream<32, MODE, E>(ctx, sp, smem, grid);
    }
    return fail(ctx, GANREV_EINVAL, "bad NQ %d", NQ);
}
static int stream_nq(int nq) { return nq <= 4 ? 4 : (nq <= 8 ? 8 : (nq <= 16 ? 16 : (nq <= 24 ? 24 : 32))); }

// ---- register-tiled labelling kernels (kmeans / cosine-min, 9 <= nq <= 32, d % 4 == 0, d <= 128): plan + launch
static bool rtile_plan(ganrev_ctx* ctx, const scan::ScanParams& p, int NQ, int mode, scan::StreamParams& sp, size_t& smem, int& grid) {
    if (!ctx->rtile || p.nq <= 8 || p.nq > 32 || p.d % 4 != 0 || p.d > 128) return false;
    const int T = NQ * 8, S = scan::wide4_stride(p.d), NW = NQ / 4;
    sp.s = p;
    sp.groups = mode == 1 ? std::max(1, T / (p.d / 4)) : 0;
    smem = sizeof(float) * (static_cast<size_t>(scan::SR + NQ) * S + 2 * static_cast<size_t>(scan::SR) * NW + 2 * scan::SR + NQ + 2) +
           (mode == 1 ? sizeof(unsigned long long) * (static_cast<size_t>(p.nq) * p.d + p.nq) : 0);
    if (smem > 200 * 1024) return false;
    const int per_sm = std::max<int>(1, std::min<int>({4, static_cast<int>((220 * 1024) / (smem + 1024)), 2048 / T}));
    const long long n_tiles = (p.n_rows + scan::SR - 1) / scan::SR;
    grid = static_cast<int>(std::max<long long>(1, std::min<long long>(n_tiles, static_cast<long long>(ctx->num_sms) * per_sm)));
    sp.tiles_per_block = (n_tiles + grid - 1) / grid;
    grid = static_cast<int>(std::max<long long>(1, (n_tiles + sp.tiles_per_block - 1) / sp.tiles_per_block));
    return true;
}
template <int NQ, int MODE>
static int launch_rtile(ganrev_ctx* ctx, const scan::StreamParams& sp, size_t smem, int grid) {
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(scan::rtile_kernel<NQ, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        CU_TRY(cudaFuncSetAttribute(scan::rtile_kernel<NQ, MODE>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr_max = smem;
    }
    scan::rtile_kernel<NQ, MODE><<<grid, NQ * 8, smem, ctx->stream>>>(sp);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}
template <int MODE>
static int dispatch_rtile(ganrev_ctx* ctx, int NQ, const scan::StreamParams& sp, size_t smem, int grid) {
    switch (NQ) {
        case 16: return launch_rtile<16, MODE>(ctx, sp, smem, grid);
        case 24: return launch_rtile<24, MODE>(ctx, sp, smem, grid);
        case 32: return launch_rtile<32, MODE>(ctx, sp, smem, grid);
    }
    return fail(ctx, GANREV_EINVAL, "bad NQ %d", NQ);
}

// ---- tensor-core labelling (label_tc.cuh): kmeans (MODE 1) / cosine-min (MODE 2) for k <= 32, d % 4 == 0, d <= 128
static size_t label_tc_smem(const scan::ScanParams& p, int mode) {
    const int d = p.d, nsl = (d + 63) / 64;
    return static_cast<size_t>(nsl) * 2 * ltc::kABlk + static_cast<size_t>(nsl) * 2 * ltc::kBBlk + 2 * static_cast<size_t>(ltc::LR) * scan::wide4_stride(d) * 4 + 32 + 64 * 4 +
           (3 * ltc::LR + 36 + 128) * 4 + 16 + ltc::kAmbStage * 4 + (mode == 2 ? ltc::LN * (d | 1) * 4 : 0) + 8 + (mode == 1 ? (static_cast<size_t>(p.nq) * d + p.nq) * 8 : 0) + 1024 + 64;
}
static bool label_tc_ok(const ganrev_ctx* ctx, const scan::ScanParams& p, int mode) {
    return ctx->label_tc && p.nq >= 1 && p.nq <= 32 && p.d % 4 == 0 && p.d <= 128 && p.n_rows > 0 && label_tc_smem(p, mode) <= 227 * 1024;
}
template <int MODE>
static int launch_label_tc(ganrev_ctx* ctx, const scan::ScanParams& p) {
    RC_TRY(ensure(ctx, ctx->amb, sizeof(unsigned) * (static_cast<size_t>(p.n_rows) + 4)));
    unsigned* d_count = static_cast<unsigned*>(ctx->amb.p);
    unsigned* d_rows = d_count + 4;
    CU_TRY(cudaMemsetAsync(d_count, 0, sizeof(unsigned), ctx->stream));
    ltc::LabelParams lp{};
    lp.s = p; lp.n_tiles = (p.n_rows + ltc::LR - 1) / ltc::LR; lp.amb_rows = d_rows; lp.amb_count = d_count; lp.err_flag = ctx->d_err_flag; lp.dbg = ctx->dbg >> 8;
    const size_t smem = label_tc_smem(p, MODE);
    static size_t attr_max_dev[kMaxDevices] = {};
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(ltc::label_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    const int per_sm = smem <= 110 * 1024 ? 2 : 1;
    const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(lp.n_tiles, static_cast<long long>(ctx->num_sms) * per_sm)));
    ltc::label_tc_kernel<MODE><<<grid, ltc::kThreads, smem, ctx->stream>>>(lp);
    ltc::label_exact_list_kernel<MODE><<<2 * ctx->num_sms, 256, 0, ctx->stream>>>(p, d_rows, d_count);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

// ---- TMA -> tf32 tcgen05 filter pipeline (stream_tc.cuh): search (MODE 0), kmeans (MODE 1), cosine-min (MODE 2) for nq <= 32, d % 4 == 0
static int tfs_nqp(int nq) { return nq <= 16 ? 16 : 32; }
static bool tfs_plan(const ganrev_ctx* ctx, const scan::ScanParams& p, int mode, int K2, tfs::TfsParams& tp, size_t& smem, int& grid) {
    if (!ctx->stream_tc || p.nq < 1 || p.nq > 32 || p.d % 4 != 0 || p.d < 4 || p.n_rows < 1 || p.n_rows > 0x7fffff00LL) return false;
    if ((reinterpret_cast<uintptr_t>(p.db) & 15) != 0) return false;
    const int NQP = tfs_nqp(p.nq);
    const int nbox = (p.d + tfs::kBoxCols - 1) / tfs::kBoxCols;
    const size_t budget = 227 * 1024;
    // the chains' fp32 centroid copy lives in shared memory unless that leaves fewer than three tiles of ring slots
    bool cen_global = false;
    size_t fixed = tfs::tfs_fixed_bytes(mode, NQP, K2, p.nq, p.d, false) + 1024;
    if (fixed > budget || (budget - fixed) / tfs::kSlotBytes < static_cast<size_t>(std::min(mode == 0 ? 8 : 3 * nbox, tfs::kMaxSlots))) {
        cen_global = true;
        fixed = tfs::tfs_fixed_bytes(mode, NQP, K2, p.nq, p.d, true) + 1024;
    }
    if (fixed + 4 * static_cast<size_t>(tfs::kSlotBytes) > budget) return false;
    int nslots = static_cast<int>(std::min<size_t>(tfs::kMaxSlots, (budget - fixed) / tfs::kSlotBytes));
    tp.cen_global = cen_global ? 1 : 0;
    if (mode != 0 && nslots < nbox + 1) return false;            // a tile stays resident until its rows were consumed
    if (mode == 1 && (p.d / 4 > tfs::kSumThreads || p.nq > 2 * tfs::kLPT * (tfs::kSumThreads / (p.d / 4)))) return false;   // the sums live in registers: kLPT (or 2 kLPT) labels per thread
    if (mode != 0 && nslots >= 2 * nbox) nslots = std::min(nslots, 3 * nbox);   // three tiles in flight are plenty
    tp.s = p;
    tp.n_tiles = (p.n_rows + tfs::kRows - 1) / tfs::kRows;
    tp.nbox = nbox; tp.nslots = nslots; tp.err_flag = ctx->d_err_flag; tp.dbg = ctx->dbg >> 16;
    tp.trace = (ctx->trace.p && ctx->trace_layer == "tfs") ? static_cast<long long*>(ctx->trace.p) : nullptr;
    smem = fixed + static_cast<size_t>(nslots) * tfs::kSlotBytes;
    grid = static_cast<int>(std::max<long long>(1, std::min<long long>(tp.n_tiles, ctx->num_sms)));
    return true;
}
static int tfs_make_map(ganrev_ctx* ctx, CUtensorMap* m, const float* base, int d, long long rows) {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(d), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(d) * 4};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(tfs::kBoxCols), static_cast<cuuint32_t>(tfs::kRows)};
    const cuuint32_t es[2] = {1u, 1u};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, GANREV_ECUDA, "cuTensorMapEncodeTiled(database rows) failed: %d", (int)r);
    return GANREV_OK;
}
template <int MODE, int NQP, int E>
static int launch_tfs_one(ganrev_ctx* ctx, const CUtensorMap& tm, const tfs::TfsParams& tp, size_t smem, int grid) {
    static size_t attr_max_dev[kMaxDevices] = {};
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(tfs::tfs_kernel<MODE, NQP, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    tfs::tfs_kernel<MODE, NQP, E><<<grid, tfs::threads_of<MODE>(), smem, ctx->stream>>>(tm, tp);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}
template <int MODE, int E>
static int launch_tfs(ganrev_ctx* ctx, tfs::TfsParams& tp, size_t smem, int grid) {
    const scan::ScanParams& p = tp.s;
    CUtensorMap tm;
    RC_TRY(tfs_make_map(ctx, &tm, p.db, p.d, p.n_rows));
    if (!ctx->tfs_aux.p) {
        RC_TRY(ensure(ctx, ctx->tfs_aux, 32 * sizeof(unsigned) + 4 * sizeof(unsigned long long)));
        CU_TRY(cudaMemsetAsync(ctx->tfs_aux.p, 0, 32 * sizeof(unsigned) + 4 * sizeof(unsigned long long), ctx->stream));
    }
    tp.gthr = static_cast<unsigned*>(ctx->tfs_aux.p);
    tp.stats = reinterpret_cast<unsigned long long*>(tp.gthr + 32);
    if (MODE == 0) CU_TRY(cudaMemsetAsync(tp.gthr, 0, 32 * sizeof(unsigned), ctx->stream));
    if (MODE != 0) {
        RC_TRY(ensure(ctx, ctx->amb, sizeof(unsigned) * (static_cast<size_t>(p.n_rows) + 4)));
        tp.amb_count = static_cast<unsigned*>(ctx->amb.p);
        tp.amb_rows = tp.amb_count + 4;
        CU_TRY(cudaMemsetAsync(tp.amb_count, 0, sizeof(unsigned), ctx->stream));
    }
    ctx->tfs_launches++;
    if (tfs_nqp(p.nq) == 16) RC_TRY((launch_tfs_one<MODE, 16, E>(ctx, tm, tp, smem, grid)));
    else RC_TRY((launch_tfs_one<MODE, 32, E>(ctx, tm, tp, smem, grid)));
    if (MODE != 0) {
        ltc::label_exact_list_kernel<(MODE == 0 ? 1 : MODE)><<<2 * ctx->num_sms, 256, 0, ctx->stream>>>(p, tp.amb_rows, tp.amb_count);
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    return GANREV_OK;
}

// merge the per-split lists, (multi-GPU) allgather + merge across ranks, copy results out
static int search_finish(ganrev_ctx* ctx, const unsigned long long* partial, int splits, int Q, int k, int64_t* ids, float* scores) {
    const unsigned mblocks = static_cast<unsigned>((static_cast<long long>(Q) * 32 + scan::kThreads - 1) / scan::kThreads);
    const bool multi = ctx->world > 1;
    if (multi) {
        RC_TRY(ensure(ctx, ctx->keys, sizeof(unsigned long long) * static_cast<size_t>(Q) * k));
        RC_TRY(ensure(ctx, ctx->keys_all, sizeof(unsigned long long) * static_cast<size_t>(Q) * k * ctx->world));
    }
    {
        ProfScope ps(ctx, "search_merge", 0.0, 8.0 * splits * Q * k + 12.0 * Q * k);
        if (k <= 32)
            scan::merge_kernel<1><<<mblocks, scan::kThreads, 0, ctx->stream>>>(partial, splits, Q, k, ctx->db_offset, multi ? 1 : 0,
                static_cast<long long*>(ctx->ids.p), static_cast<float*>(ctx->scores.p), static_cast<unsigned long long*>(ctx->keys.p));
        else
            scan::merge_kernel<4><<<mblocks, scan::kThreads, 0, ctx->stream>>>(partial, splits, Q, k, ctx->db_offset, multi ? 1 : 0,
                static_cast<long long*>(ctx->ids.p), static_cast<float*>(ctx->scores.p), static_cast<unsigned long long*>(ctx->keys.p));
        CU_TRY(cudaGetLastError());
    }
    if (multi) {
        // per-query top-k allgather (Q*k*8 B per rank), then the same merge over `world` partial lists
        {
            ProfScope pc(ctx, "nccl_allgather_topk", 0.0, 8.0 * ctx->world * Q * k, false);
            NCCL_TRY(ctx->nccl.AllGather(ctx->keys.p, ctx->keys_all.p, static_cast<size_t>(Q) * k, ncclUint64, ctx->comm, ctx->stream));
        }
        ProfScope ps(ctx, "search_merge_global", 0.0, 8.0 * ctx->world * Q * k + 12.0 * Q * k);
        if (k <= 32)
            scan::merge_kernel<1><<<mblocks, scan::kThreads, 0, ctx->stream>>>(static_cast<const unsigned long long*>(ctx->keys_all.p), ctx->world, Q, k, 0, 0,
                static_cast<long long*>(ctx->ids.p), static_cast<float*>(ctx->scores.p), nullptr);
        else
            scan::merge_kernel<4><<<mblocks, scan::kThreads, 0, ctx->stream>>>(static_cast<const unsigned long long*>(ctx->keys_all.p), ctx->world, Q, k, 0, 0,
                static_cast<long long*>(ctx->ids.p), static_cast<float*>(ctx->scores.p), nullptr);
        CU_TRY(cudaGetLastError());
    }
    CU_TRY(cudaMemcpyAsync(ids, ctx->ids.p, sizeof(long long) * static_cast<size_t>(Q) * k, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaMemcpyAsync(scores, ctx->scores.p, sizeof(float) * static_cast<size_t>(Q) * k, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}


// queries already on the device in ctx->q (Q x d), their 1/(|q|^2+eps) in ctx->rq: the fmaf-chain kernels
static int search_exact_dev(ganrev_ctx* ctx, int Q, int k, int64_t* ids, float* scores) {
    const int d = ctx->db_d;
    const int64_t N = ctx->db_n;
    if (Q <= 32 && k <= 128) {     // HBM-bound regime, tensor-core filter: the database streams once through TMA, chains only for candidates
        scan::ScanParams p{};
        p.db = ctx->db_ptr; p.rdb = static_cast<const float*>(ctx->rdb.p); p.n_rows = N; p.d = d;
        p.q = static_cast<const float*>(ctx->q.p); p.rq = static_cast<const float*>(ctx->rq.p); p.nq = Q; p.k = k;
        tfs::TfsParams tp{};
        size_t smem = 0;
        int grid = 0;
        if (tfs_plan(ctx, p, 0, k <= 32 ? 32 : 128, tp, smem, grid)) {
            RC_TRY(ensure(ctx, ctx->partial, sizeof(unsigned long long) * static_cast<size_t>(grid) * Q * k));
            RC_TRY(ensure(ctx, ctx->ids, sizeof(long long) * static_cast<size_t>(Q) * k));
            RC_TRY(ensure(ctx, ctx->scores, sizeof(float) * static_cast<size_t>(Q) * k));
            tp.s.partial = static_cast<unsigned long long*>(ctx->partial.p);
            {
                ProfScope ps(ctx, "search_scan", 2.0 * N * Q * d, 4.0 * N * d + 4.0 * Q * d + 8.0 * grid * Q * k);
                if (k <= 32) RC_TRY((launch_tfs<0, 1>(ctx, tp, smem, grid))); else RC_TRY((launch_tfs<0, 4>(ctx, tp, smem, grid)));
            }
            return search_finish(ctx, tp.s.partial, grid, Q, k, ids, scores);
        }
    }
    if (Q <= 16 && d % 4 == 0) {   // HBM-bound regime: stream the database once
        scan::ScanParams p{};
        p.db = ctx->db_ptr; p.rdb = static_cast<const float*>(ctx->rdb.p); p.n_rows = N; p.d = d;
        p.q = static_cast<const float*>(ctx->q.p); p.rq = static_cast<const float*>(ctx->rq.p); p.nq = Q; p.k = k;
        scan::StreamParams sp{};
        size_t smem = 0;
        int grid = 0;
        const int NQ = stream_nq(Q), K2 = k <= 32 ? 32 : 128;
        if (stream_plan(ctx, p, NQ, 0, K2, sp, smem, grid)) {
            RC_TRY(ensure(ctx, ctx->partial, sizeof(unsigned long long) * static_cast<size_t>(grid) * Q * k));
            RC_TRY(ensure(ctx, ctx->ids, sizeof(long long) * static_cast<size_t>(Q) * k));
            RC_TRY(ensure(ctx, ctx->scores, sizeof(float) * static_cast<size_t>(Q) * k));
            sp.s.partial = static_cast<unsigned long long*>(ctx->partial.p);
            {
                ProfScope ps(ctx, "search_scan", 2.0 * N * Q * d, 4.0 * N * d + 4.0 * Q * d + 8.0 * grid * Q * k);
                if (k <= 32) RC_TRY((dispatch_stream<0, 1>(ctx, NQ, sp, smem, grid))); else RC_TRY((dispatch_stream<0, 4>(ctx, NQ, sp, smem, grid)));
            }
            return search_finish(ctx, sp.s.partial, grid, Q, k, ids, scores);
        }
    }
    const int TQ = Q <= 16 ? 1 : 4;
    const int QT = 16 * TQ;
    const int qtiles = (Q + QT - 1) / QT;
    // row splits: fill the machine about 4 blocks per SM deep, at least one 128-row tile each
    const int64_t row_tiles = std::max<int64_t>(1, (N + scan::RT - 1) / scan::RT);
    int splits = static_cast<int>(std::min<int64_t>(row_tiles, std::max<int64_t>(1, (4LL * ctx->num_sms + qtiles - 1) / qtiles)));
    const bool wide4 = TQ == 4 && d <= 128 && d % 4 == 0;
    if (wide4) {
        // two blocks of the wide kernel are resident per SM: pick the split count whose block total wastes the
        // least of its last wave (and keeps at least 8 row tiles per split so the top-k lists warm up once)
        const int64_t R = 2LL * ctx->num_sms;
        double best = 1e30;
        for (int m = 2; m <= 16; ++m) {
            const int64_t sp = std::min<int64_t>(std::max<int64_t>(1, row_tiles / 8), std::max<int64_t>(1, m * R / qtiles));
            const int64_t total = sp * qtiles, waves = (total + R - 1) / R;
            const double waste = static_cast<double>(waves * R) / static_cast<double>(total) + 0.002 * m;   // mild preference for fewer, longer splits
            if (waste < best) { best = waste; splits = static_cast<int>(sp); }
        }
    }
    const int64_t rows_per_split = ((row_tiles + splits - 1) / splits) * scan::RT;
    splits = static_cast<int>(std::max<int64_t>(1, (N + rows_per_split - 1) / rows_per_split));
    RC_TRY(ensure(ctx, ctx->partial, sizeof(unsigned long long) * static_cast<size_t>(splits) * Q * k));
    RC_TRY(ensure(ctx, ctx->ids, sizeof(long long) * static_cast<size_t>(Q) * k));
    RC_TRY(ensure(ctx, ctx->scores, sizeof(float) * static_cast<size_t>(Q) * k));
    scan::ScanParams p{};
    p.db = ctx->db_ptr; p.rdb = static_cast<const float*>(ctx->rdb.p); p.n_rows = N; p.d = d;
    p.q = static_cast<const float*>(ctx->q.p); p.rq = static_cast<const float*>(ctx->rq.p); p.nq = Q; p.k = k;
    p.partial = static_cast<unsigned long long*>(ctx->partial.p); p.rows_per_split = rows_per_split;
    {
        ProfScope ps(ctx, "search_scan", 2.0 * N * Q * d, 4.0 * N * d + 4.0 * Q * d + 8.0 * splits * Q * k);
        const bool wide = TQ == 4 && d <= 128;
        if (TQ == 1)   { if (k <= 32) RC_TRY((launch_search<1, 1>(ctx, p, splits))); else RC_TRY((launch_search<1, 4>(ctx, p, splits))); }
        else if (wide && p.d % 4 == 0) { if (k <= 32) RC_TRY((launch_search_wide4<1>(ctx, p, splits))); else RC_TRY((launch_search_wide4<4>(ctx, p, splits))); }
        else if (wide) { if (k <= 32) RC_TRY((launch_search_wide<1>(ctx, p, splits))); else RC_TRY((launch_search_wide<4>(ctx, p, splits))); }
        else           { if (k <= 32) RC_TRY((launch_search<4, 1>(ctx, p, splits))); else RC_TRY((launch_search<4, 4>(ctx, p, splits))); }
    }
    return search_finish(ctx, p.partial, splits, Q, k, ids, scores);
}

// ---- tensor-core candidate filter + exact re-score (search_tc.cuh)
static int tc_make_map(ganrev_ctx* ctx, CUtensorMap* m, const void* base, int kp, long long rows, long long row_pitch_elems, int box_rows) {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(kp), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(row_pitch_elems) * 2};
    const cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t es[2] = {1u, 1u};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, GANREV_ECUDA, "cuTensorMapEncodeTiled(search operand) failed: %d", (int)r);
    return GANREV_OK;
}
static int tc_pack(ganrev_ctx* ctx, const char* name, const float* x, const float* rn, int64_t n, int d, DevBuf& out, bool is_query) {
    const int kp = stc::packed_cols(d);
    RC_TRY(ensure(ctx, out, sizeof(bf16) * static_cast<size_t>(std::max<int64_t>(n, 1)) * kp));
    RC_TRY(ensure(ctx, ctx->tc_special, sizeof(unsigned) * (stc::kMaxSpecial + 4)));
    RC_TRY(ensure(ctx, ctx->tc_flags, 4 * sizeof(int)));
    unsigned* sp_rows = static_cast<unsigned*>(ctx->tc_special.p);
    unsigned* sp_count = sp_rows + stc::kMaxSpecial;
    int* flags = static_cast<int*>(ctx->tc_flags.p);           // [0] this search, [1] the database
    if (!is_query) { CU_TRY(cudaMemsetAsync(sp_count, 0, sizeof(unsigned), ctx->stream)); CU_TRY(cudaMemsetAsync(flags + 1, 0, sizeof(int), ctx->stream)); }
    ProfScope ps(ctx, name, 2.0 * n * d, n * (4.0 * d + 2.0 * kp));
    const long long tot = n * (kp / 4);
    if (tot > 0) stc::pack_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, ctx->stream>>>(x, rn, n, d, static_cast<bf16*>(out.p), is_query ? 1 : 0,
                                                                                                 sp_rows, sp_count, is_query ? flags : flags + 1);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}
struct TcPlan { int levels; int stride[8]; int cap; };
__global__ void tc_combine_flags_kernel(int* flags, int extra) { flags[2] = flags[0] | flags[1] | extra; }
static bool tc_plan(const ganrev_ctx* ctx, int Q, int k, TcPlan& pl) {
    const int64_t N = ctx->db_n;
    if (N < 8192) return false;
    const int64_t n_t = std::max<int64_t>(1024, 8LL * k);      // rows of the coarsest (exhaustively re-scored) sample
    const int64_t sL = N / n_t;                                 // >= 8
    const int L = std::max(1, static_cast<int>(std::ceil(std::log(static_cast<double>(sL)) / std::log(24.0) - 1e-9)));   // levels at most 24x apart: ~24 k candidates per query against lists of >= 64 k
    if (L > 6) return false;
    const double r = std::pow(static_cast<double>(sL), 1.0 / L);
    pl.levels = L;
    pl.stride[0] = 1;
    for (int i = 1; i <= L; ++i) {
        int s = i == L ? static_cast<int>(sL) : static_cast<int>(std::llround(std::pow(r, i)));
        pl.stride[i] = std::max(s, pl.stride[i - 1] + 1);
    }
    pl.cap = std::max(2048, 64 * k);
    return true;
}
// Runs the levels on this rank's shard: leaves the shard's top-k keys in ctx->partial and the flags on the device.
static int search_tc_local(ganrev_ctx* ctx, const TcPlan& pl, int Q, int k) {
    const int d = ctx->db_d, kp = stc::packed_cols(d);
    const int64_t N = ctx->db_n;
    int* d_flags = static_cast<int*>(ctx->tc_flags.p);
    if (!ctx->pdb_valid) {
        RC_TRY(tc_pack(ctx, "search_tc_pack_db", ctx->db_ptr, static_cast<const float*>(ctx->rdb.p), N, d, ctx->pdb, false));
        ctx->pdb_valid = true;
    }
    RC_TRY(tc_pack(ctx, "search_tc_pack_q", static_cast<const float*>(ctx->q.p), static_cast<const float*>(ctx->rq.p), Q, d, ctx->pq, true));
    RC_TRY(ensure(ctx, ctx->tc_thr, sizeof(float) * Q));
    // per level: cnt[Q] | offsets[Q] | cursor[Q] | total; pairs in arrival order, then candidates grouped by query
    const size_t pair_cap = static_cast<size_t>(Q) * std::max(2048, 100 * k);
    RC_TRY(ensure(ctx, ctx->tc_cnt, sizeof(unsigned) * (3 * static_cast<size_t>(Q) + 4)));
    RC_TRY(ensure(ctx, ctx->tc_pairs, sizeof(uint4) * pair_cap));
    RC_TRY(ensure(ctx, ctx->tc_cand, 2 * sizeof(unsigned) * pair_cap));          // rows, then their approximate scores
    RC_TRY(ensure(ctx, ctx->tc_keys, sizeof(unsigned long long) * static_cast<size_t>(Q) * k));
    unsigned* d_cnt = static_cast<unsigned*>(ctx->tc_cnt.p);
    unsigned* d_off = d_cnt + Q;
    unsigned* d_cur = d_off + Q;
    unsigned* d_total = d_cur + Q;
    unsigned* sp_rows = static_cast<unsigned*>(ctx->tc_special.p);
    static size_t attr_dev[kMaxDevices][2] = {};
    if (!attr_dev[ctx->device][0]) {
        CU_TRY(cudaFuncSetAttribute(stc::filter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, stc::kSmem));
        CU_TRY(cudaFuncSetAttribute(stc::filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, stc::kSmem));
        attr_dev[ctx->device][0] = 1;
    }
    const int64_t nL = (N + pl.stride[pl.levels] - 1) / pl.stride[pl.levels];
    const size_t rs_smem = 12 * (static_cast<size_t>(std::max<int64_t>(pl.cap, nL)) + stc::kMaxSpecial + 8) + 4 * static_cast<size_t>(d) + 64;
    if (rs_smem > attr_dev[ctx->device][1]) {
        CU_TRY(cudaFuncSetAttribute(stc::rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(rs_smem)));
        attr_dev[ctx->device][1] = rs_smem;
    }
    stc::RescoreParams rp{};
    rp.db = ctx->db_ptr; rp.rdb = static_cast<const float*>(ctx->rdb.p); rp.n = N; rp.d = d;
    rp.q = static_cast<const float*>(ctx->q.p); rp.rq = static_cast<const float*>(ctx->rq.p); rp.nq = Q; rp.k = k;
    rp.cnt = d_cnt; rp.offsets = d_off; rp.cand = static_cast<const unsigned*>(ctx->tc_cand.p);
    rp.cand_score = reinterpret_cast<const float*>(static_cast<const unsigned*>(ctx->tc_cand.p) + pair_cap); rp.cap = pl.cap;
    rp.special_rows = sp_rows; rp.special_count = sp_rows + stc::kMaxSpecial; rp.eps = stc::tc_eps(d); rp.flags = d_flags;
    CUtensorMap tmQ, tmX;
    RC_TRY(tc_make_map(ctx, &tmQ, ctx->pq.p, kp, Q, kp, stc::QM));
    const float* d_cscore = reinterpret_cast<const float*>(static_cast<const unsigned*>(ctx->tc_cand.p) + pair_cap);
    for (int lvl = pl.levels; lvl >= 0; --lvl) {
        const int stride = pl.stride[lvl];
        const int64_t n_l = (N + stride - 1) / stride;
        const bool coarsest = lvl == pl.levels, final_level = lvl == 0;
        CU_TRY(cudaMemsetAsync(ctx->tc_cnt.p, 0, sizeof(unsigned) * (3 * static_cast<size_t>(Q) + 4), ctx->stream));
        if (coarsest) {   // every pair of the coarsest sample is kept: dense approximate scores, no pair passes the (infinite) threshold
            RC_TRY(ensure(ctx, ctx->tc_dump, sizeof(float) * static_cast<size_t>(Q) * n_l));
            CU_TRY(cudaMemsetAsync(ctx->tc_thr.p, 0x7f, sizeof(float) * Q, ctx->stream));
        }
        RC_TRY(tc_make_map(ctx, &tmX, ctx->pdb.p, kp, n_l, static_cast<long long>(stride) * kp, stc::RN));
        stc::FilterParams fp{};
        fp.nq = Q; fp.n_rows = n_l; fp.stride = stride; fp.d = d; fp.nslices = kp / 128;
        fp.q_tiles = (Q + stc::QM - 1) / stc::QM;
        fp.items = static_cast<long long>(fp.q_tiles) * ((n_l + stc::RN - 1) / stc::RN);
        fp.thr = static_cast<const float*>(ctx->tc_thr.p); fp.cnt = d_cnt;
        fp.pairs = static_cast<uint4*>(ctx->tc_pairs.p); fp.total = d_total; fp.pair_cap = static_cast<unsigned>(pair_cap);
        fp.flags = d_flags; fp.err_flag = ctx->d_err_flag; fp.dump = coarsest ? static_cast<float*>(ctx->tc_dump.p) : nullptr;
        {
            // executed work: three bf16 product chains over the 16-padded columns; bytes: the packed rows once (L2 serves the other query tiles)
            ProfScope ps(ctx, "search_tc_filter", 3.0 * 2.0 * n_l * Q * ((d + 15) / 16 * 16), 2.0 * kp * (static_cast<double>(n_l) + Q));
            const int grid = static_cast<int>(std::min<long long>(fp.items, ctx->num_sms));
            if (coarsest) stc::filter_kernel<true><<<grid, stc::kThr, stc::kSmem, ctx->stream>>>(tmQ, tmX, fp);
            else stc::filter_kernel<false><<<grid, stc::kThr, stc::kSmem, ctx->stream>>>(tmQ, tmX, fp);
            CU_TRY(cudaGetLastError());
        }
        if (!coarsest) {
            ProfScope ps(ctx, "search_tc_group", 0.0, 20.0 * Q * 32.0 * k);
            ctx->launches++;
            stc::offsets_kernel<<<1, 1024, 0, ctx->stream>>>(d_cnt, Q, static_cast<unsigned>(pl.cap), d_off, d_cur, d_flags);
            stc::scatter_kernel<<<4 * ctx->num_sms, 256, 0, ctx->stream>>>(static_cast<const uint4*>(ctx->tc_pairs.p), d_total, static_cast<unsigned>(pair_cap), d_off, d_cur,
                                                                          static_cast<unsigned*>(ctx->tc_cand.p), const_cast<float*>(d_cscore), d_flags);
            CU_TRY(cudaGetLastError());
        }
        rp.implicit_stride = coarsest ? stride : 0;
        rp.n_implicit = coarsest ? static_cast<int>(n_l) : 0;
        rp.cand_score = coarsest ? static_cast<const float*>(ctx->tc_dump.p) : d_cscore;
        rp.final_level = final_level ? 1 : 0;
        rp.next_ratio = final_level ? 1.0f : static_cast<float>(stride) / static_cast<float>(pl.stride[lvl - 1]);
        rp.keys_out = static_cast<unsigned long long*>(ctx->partial.p);
        rp.thr_out = final_level ? nullptr : static_cast<float*>(ctx->tc_thr.p);
        ProfScope ps(ctx, final_level ? "search_tc_rescore" : "search_tc_select", final_level ? 2.0 * Q * d * 1.5 * k : 0.0, 0.0);
        stc::rescore_kernel<<<Q, 256, rs_smem, ctx->stream>>>(rp);
        CU_TRY(cudaGetLastError());
    }
    return GANREV_OK;
}
// *served = true: ids / scores are final.  *served = false: the caller runs the fmaf-chain kernels (on every rank alike).
static int search_tc_dev(ganrev_ctx* ctx, int Q, int k, int64_t* ids, float* scores, bool* served) {
    *served = false;
    // eligibility from quantities every rank agrees on (the branches below contain collectives)
    if (!ctx->search_tc || Q < 48 || k > 128 || ctx->db_d > 1024 || ctx->db_total < 8192LL * ctx->world) return GANREV_OK;
    TcPlan pl;
    const bool local_ok = tc_plan(ctx, Q, k, pl);
    RC_TRY(ensure(ctx, ctx->tc_flags, 4 * sizeof(int)));
    RC_TRY(ensure(ctx, ctx->partial, sizeof(unsigned long long) * static_cast<size_t>(Q) * k));
    RC_TRY(ensure(ctx, ctx->ids, sizeof(long long) * static_cast<size_t>(Q) * k));
    RC_TRY(ensure(ctx, ctx->scores, sizeof(float) * static_cast<size_t>(Q) * k));
    int* d_flags = static_cast<int*>(ctx->tc_flags.p);           // [0] this search, [1] the database, [2] combined over ranks
    CU_TRY(cudaMemsetAsync(d_flags, 0, sizeof(int), ctx->stream));
    if (local_ok) RC_TRY(search_tc_local(ctx, pl, Q, k));
    int h_flags[2] = {0, 0};
    if (ctx->world == 1) {
        if (!local_ok) return GANREV_OK;
        // optimistic: merge and copy the result out, then look at the flags (no extra synchronisation on the common path)
        RC_TRY(search_finish(ctx, static_cast<const unsigned long long*>(ctx->partial.p), 1, Q, k, ids, scores));
        CU_TRY(cudaMemcpy(h_flags, d_flags, 2 * sizeof(int), cudaMemcpyDeviceToHost));
    } else {
        // every rank must take the same branch: combine the flags first (a shard too small for the levels votes for the fallback)
        tc_combine_flags_kernel<<<1, 1, 0, ctx->stream>>>(d_flags, local_ok ? 0 : stc::FLAG_OVERFLOW);
        ctx->launches++;
        NCCL_TRY(ctx->nccl.AllReduce(d_flags + 2, d_flags + 2, 1, ncclInt32, ncclMax, ctx->comm, ctx->stream));
        CU_TRY(cudaMemcpyAsync(h_flags, d_flags + 2, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        RC_TRY(finish(ctx));
        if (h_flags[0] == 0) RC_TRY(search_finish(ctx, static_cast<const unsigned long long*>(ctx->partial.p), 1, Q, k, ids, scores));
    }
    if (h_flags[0] | h_flags[1]) { ctx->tc_fallbacks++; return GANREV_OK; }   // overflow / special vectors: the fmaf-chain kernels decide
    ctx->tc_searches++;
    *served = true;
    return GANREV_OK;
}

static int search_dev(ganrev_ctx* ctx, int Q, int k, int64_t* ids, float* scores) {
    RC_TRY(ensure(ctx, ctx->rq, sizeof(float) * Q));
    RC_TRY(vec_prep(ctx, static_cast<const float*>(ctx->q.p), Q, ctx->db_d, static_cast<float*>(ctx->rq.p), nullptr, nullptr));
    bool served = false;
    RC_TRY(search_tc_dev(ctx, Q, k, ids, scores, &served));
    if (served) return GANREV_OK;
    return search_exact_dev(ctx, Q, k, ids, scores);
}

extern "C" {
int ganrev_search_cosine(ganrev_ctx* ctx, const float* queries, int Q, int k, int64_t* ids, float* scores) {
    if (!ctx || !queries || Q < 0 || k < 1 || k > 128 || !ids || !scores) return ctx ? fail(ctx, GANREV_EINVAL, "bad search arguments (k must be 1..128)") : GANREV_EINVAL;
    if (!ctx->db_ptr) return fail(ctx, GANREV_ESTATE, "database not set");
    if (Q == 0) return GANREV_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(ensure(ctx, ctx->q, sizeof(float) * static_cast<size_t>(Q) * ctx->db_d));
    CU_TRY(cudaMemcpyAsync(ctx->q.p, queries, sizeof(float) * static_cast<size_t>(Q) * ctx->db_d, cudaMemcpyHostToDevice, ctx->stream));
    return search_dev(ctx, Q, k, ids, scores);
}

int ganrev_search_rows(ganrev_ctx* ctx, const int64_t* rows, int Q, int k, int64_t* ids, float* scores) {
    if (!ctx || !rows || Q < 0 || k < 1 || k > 128 || !ids || !scores) return ctx ? fail(ctx, GANREV_EINVAL, "bad search_rows arguments (k must be 1..128)") : GANREV_EINVAL;
    if (!ctx->db_ptr) return fail(ctx, GANREV_ESTATE, "database not set");
    if (Q == 0) return GANREV_OK;
    for (int i = 0; i < Q; ++i)
        if (rows[i] < 0 || rows[i] >= ctx->db_total) return fail(ctx, GANREV_EINVAL, "row id %lld outside the database", (long long)rows[i]);
    CU_TRY(cudaSetDevice(ctx->device));
    const int d = ctx->db_d;
    RC_TRY(ensure(ctx, ctx->q, sizeof(float) * static_cast<size_t>(Q) * d));
    RC_TRY(ensure(ctx, ctx->stage_b, sizeof(long long) * static_cast<size_t>(Q)));
    CU_TRY(cudaMemcpyAsync(ctx->stage_b.p, rows, sizeof(long long) * Q, cudaMemcpyHostToDevice, ctx->stream));
    {
        ProfScope ps(ctx, "gather_rows", 0.0, 8.0 * Q * d);
        const long long tot = static_cast<long long>(Q) * d;
        scan::gather_rows_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, ctx->stream>>>(
            ctx->db_ptr, ctx->db_n, d, ctx->db_offset, static_cast<const long long*>(ctx->stage_b.p), Q, static_cast<float*>(ctx->q.p));
        CU_TRY(cudaGetLastError());
    }
    if (ctx->world > 1) {   // exactly one rank holds each row; the others contribute +0.0f (all-zero bits)
        ProfScope pc(ctx, "nccl_allreduce_queries", 0.0, 4.0 * Q * d, false);
        NCCL_TRY(ctx->nccl.AllReduce(ctx->q.p, ctx->q.p, static_cast<size_t>(Q) * d, ncclUint32, ncclMax, ctx->comm, ctx->stream));
    }
    return search_dev(ctx, Q, k, ids, scores);
}
}  // extern "C"
template <int TQ, int MODE>
static int launch_assign(ganrev_ctx* ctx, const scan::ScanParams& p) {
    constexpr int QT = 16 * TQ;
    size_t smem = sizeof(float) * (scan::DK * scan::XS + scan::DK * QT + 16 * scan::RT) + sizeof(int) * (16 * scan::RT + scan::RT);
    if (MODE == 1 && p.smem_acc) smem += sizeof(unsigned long long) * (static_cast<size_t>(p.nq) * p.d + p.nq);
    static size_t attr_max_dev[kMaxDevices] = {};          // function attributes are per device
    size_t& attr_max = attr_max_dev[ctx->device];
    if (smem > attr_max) {
        CU_TRY(cudaFuncSetAttribute(scan::assign_kernel<TQ, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr_max = smem;
    }
    const long long n_tiles = (p.n_rows + scan::RT - 1) / scan::RT;
    const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(n_tiles, 4LL * ctx->num_sms)));
    scan::assign_kernel<TQ, MODE><<<grid, scan::kThreads, smem, ctx->stream>>>(p, n_tiles);
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

// ---- kmeans labelling for k > 32 on the tensor cores (kmeans_tc.cuh)
static bool kmeans_tc_ok(const ganrev_ctx* ctx, int k) {
    return ctx->kmeans_tc && k > 32 && ctx->db_d <= 1024 && ctx->db_n >= 1 && ctx->db_ptr != nullptr;
}
static int kmeans_tc_iteration(ganrev_ctx* ctx, const scan::ScanParams& p) {
    const int d = p.d, k = p.nq, kp = stc::packed_cols(d);
    const int64_t N = p.n_rows;
    if (!ctx->pdb_valid) {
        RC_TRY(tc_pack(ctx, "search_tc_pack_db", ctx->db_ptr, static_cast<const float*>(ctx->rdb.p), N, d, ctx->pdb, false));
        ctx->pdb_valid = true;
    }
    RC_TRY(tc_pack(ctx, "kmeans_tc_pack_c", p.q, nullptr, k, d, ctx->pq, true));
    // [count2 | cm2 | pad] | near-tie entries uint4[N] | full rows u32[N] | full keys u64[N]
    const size_t amb_bytes = 32 + sizeof(uint4) * static_cast<size_t>(N) + 4 * static_cast<size_t>(N) + 8 * static_cast<size_t>(N) + 64;
    RC_TRY(ensure(ctx, ctx->amb, amb_bytes));
    unsigned* d_count = static_cast<unsigned*>(ctx->amb.p);
    float* d_cm = reinterpret_cast<float*>(d_count + 2);
    uint4* d_rows = reinterpret_cast<uint4*>(d_count + 8);
    unsigned long long* d_keys = reinterpret_cast<unsigned long long*>(d_rows + N);
    unsigned* d_full = reinterpret_cast<unsigned*>(d_keys + N);
    CU_TRY(cudaMemsetAsync(d_keys, 0, 8 * static_cast<size_t>(N), ctx->stream));   // (the layout depends on N and the buffer is shared: clear every time, 8 bytes per row)
    CU_TRY(cudaMemsetAsync(d_count, 0, 2 * sizeof(unsigned), ctx->stream));
    ktc::cmax_kernel<<<1, 32, 0, ctx->stream>>>(p.c2, k, stc::tc_eps(d), d_cm);
    static bool attr_dev[kMaxDevices] = {};
    if (!attr_dev[ctx->device]) {
        CU_TRY(cudaFuncSetAttribute(ktc::label_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ktc::kSmem));
        attr_dev[ctx->device] = true;
    }
    CUtensorMap tmX, tmC;
    RC_TRY(tc_make_map(ctx, &tmX, ctx->pdb.p, kp, N, kp, stc::QM));
    RC_TRY(tc_make_map(ctx, &tmC, ctx->pq.p, kp, k, kp, stc::RN));
    ktc::KParams kp_{};
    kp_.n_rows = N; kp_.d = d; kp_.nslices = kp / 128; kp_.k = k; kp_.nchunks = (k + stc::RN - 1) / stc::RN;
    kp_.r_tiles = (N + stc::QM - 1) / stc::QM;
    kp_.rdb = p.rdb; kp_.c2 = p.c2; kp_.cm = d_cm; kp_.labels = p.labels; kp_.amb_rows = d_rows; kp_.full_rows = d_full; kp_.amb_count = d_count; kp_.err_flag = ctx->d_err_flag;
    const int grid = static_cast<int>(std::min<long long>(kp_.r_tiles, ctx->num_sms));
    {
        ProfScope ps(ctx, "kmeans_tc_label", 3.0 * 2.0 * N * k * ((d + 15) / 16 * 16), 2.0 * kp * (static_cast<double>(N) + k));
        ktc::label_kernel<<<grid, stc::kThr, ktc::kSmem, ctx->stream>>>(tmX, tmC, kp_);
    }
    {
        ProfScope ps(ctx, "kmeans_tc_update", 1.0 * N * d, 4.0 * N * d + 4.0 * N);
        ktc::update_kernel<<<8 * ctx->num_sms, 256, 0, ctx->stream>>>(p.db, N, d, p.labels, p.sc, p.acc, p.cnt);
    }
    {
        ProfScope ps(ctx, "kmeans_tc_exact", 0.0, 0.0);
        ktc::exact_two_kernel<<<4 * ctx->num_sms, 256, 0, ctx->stream>>>(p, d_rows, d_count);
        ktc::full_scan_kernel<<<4 * ctx->num_sms, 256, 0, ctx->stream>>>(p, d_full, d_count + 1, d_keys);
        ktc::full_finalize_kernel<<<ctx->num_sms, 256, 0, ctx->stream>>>(p, d_full, d_count + 1, d_keys);
        ctx->launches += 2;
    }
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    return GANREV_OK;
}

extern "C" {
static int kmeans_shift_of(float maxabs, int64_t n_total) {
    if (!(maxabs <= 3.0e38f)) return -1;
    int e = 0;
    if (maxabs > 0.0f) (void)std::frexp(maxabs, &e);
    int n = 0;
    while ((static_cast<int64_t>(1) << n) < n_total) ++n;
    const int s = 62 - n - e;
    if (s < 0) return -1;               // llrint(x * 2^0) summed over the rows would leave int64
    return std::min(60, s);
}

int ganrev_kmeans(ganrev_ctx* ctx, int k, int niter, const float* init_centroids, float* centroids, float* total_counts, int32_t* last_labels) {
    if (!ctx || k < 1 || niter < 0 || !init_centroids || !centroids || !total_counts) return ctx ? fail(ctx, GANREV_EINVAL, "bad kmeans arguments") : GANREV_EINVAL;
    if (!ctx->db_ptr) return fail(ctx, GANREV_ESTATE, "database not set");
    CU_TRY(cudaSetDevice(ctx->device));
    const int d = ctx->db_d;
    const int64_t N = ctx->db_n;
    const int shift = kmeans_shift_of(ctx->db_maxabs, ctx->db_total);
    if (shift < 0) return fail(ctx, GANREV_EINVAL, "database contains non-finite values, or values too large for the 64-bit fixed-point centroid sums (max|x| * rows >= 2^62)");
    const double sc = std::ldexp(1.0, shift);
    const size_t kd = static_cast<size_t>(k) * d;
    RC_TRY(ensure(ctx, ctx->cen, sizeof(float) * kd));
    RC_TRY(ensure(ctx, ctx->c2, sizeof(float) * k));
    RC_TRY(ensure(ctx, ctx->acc, sizeof(unsigned long long) * (kd + k)));   // acc followed by cnt: one allreduce
    RC_TRY(ensure(ctx, ctx->total, sizeof(unsigned long long) * k));
    RC_TRY(ensure(ctx, ctx->labels, sizeof(int) * static_cast<size_t>(std::max<int64_t>(N, 1))));
    RC_TRY(ensure(ctx, ctx->tcounts, sizeof(float) * k));
    unsigned long long* d_acc = static_cast<unsigned long long*>(ctx->acc.p);
    unsigned long long* d_cnt = d_acc + kd;
    CU_TRY(cudaMemcpyAsync(ctx->cen.p, init_centroids, sizeof(float) * kd, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemsetAsync(ctx->acc.p, 0, sizeof(unsigned long long) * (kd + k), ctx->stream));
    CU_TRY(cudaMemsetAsync(ctx->total.p, 0, sizeof(unsigned long long) * k, ctx->stream));
    if (niter == 0) CU_TRY(cudaMemsetAsync(ctx->labels.p, 0xFF, sizeof(int) * static_cast<size_t>(std::max<int64_t>(N, 1)), ctx->stream));
    scan::ScanParams p{};
    p.db = ctx->db_ptr; p.rdb = static_cast<const float*>(ctx->rdb.p); p.n_rows = N; p.d = d;
    p.q = static_cast<const float*>(ctx->cen.p); p.c2 = static_cast<const float*>(ctx->c2.p); p.rq = nullptr; p.nq = k;
    p.labels = static_cast<int*>(ctx->labels.p); p.acc = d_acc; p.cnt = d_cnt; p.sc = sc;
    p.smem_acc = (kd + k) * sizeof(unsigned long long) <= 96 * 1024 ? 1 : 0;
    for (int it = 0; it < niter; ++it) {
        RC_TRY(vec_prep(ctx, static_cast<const float*>(ctx->cen.p), k, d, nullptr, static_cast<float*>(ctx->c2.p), nullptr));
        {
            ProfScope ps(ctx, "kmeans_assign", 2.0 * N * k * d + 1.0 * N * d, 8.0 * N * d + 4.0 * N + 4.0 * kd);
            scan::StreamParams sp{};
            size_t smem = 0;
            int grid = 0;
            tfs::TfsParams tp{};
            if (kmeans_tc_ok(ctx, k)) RC_TRY(kmeans_tc_iteration(ctx, p));
            else if (tfs_plan(ctx, p, 1, 0, tp, smem, grid)) {
                if (p.nq > tfs::kLPT * (tfs::kSumThreads / (p.d / 4))) RC_TRY((launch_tfs<1, 4>(ctx, tp, smem, grid)));   // more labels per sums thread
                else RC_TRY((launch_tfs<1, 1>(ctx, tp, smem, grid)));
            }
            else if (label_tc_ok(ctx, p, 1)) RC_TRY((launch_label_tc<1>(ctx, p)));
            else if (rtile_plan(ctx, p, stream_nq(k), 1, sp, smem, grid)) RC_TRY((dispatch_rtile<1>(ctx, stream_nq(k), sp, smem, grid)));
            else if (stream_plan(ctx, p, stream_nq(k), 1, 0, sp, smem, grid)) RC_TRY((dispatch_stream<1, 1>(ctx, stream_nq(k), sp, smem, grid)));
            else if (k <= 16) RC_TRY((launch_assign<1, 1>(ctx, p)));
            else RC_TRY((launch_assign<4, 1>(ctx, p)));
        }
        if (ctx->world > 1) {   // centroid sums + counts: one order-free int64 allreduce per iteration
            ProfScope pc(ctx, "nccl_allreduce_centroids", 0.0, 8.0 * (kd + k), false);
            NCCL_TRY(ctx->nccl.AllReduce(ctx->acc.p, ctx->acc.p, kd + k, ncclUint64, ncclSum, ctx->comm, ctx->stream));
        }
        {
            ProfScope ps(ctx, "kmeans_finalize", 0.0, 12.0 * kd);
            scan::kmeans_finalize_kernel<<<k, 128, 0, ctx->stream>>>(static_cast<float*>(ctx->cen.p), d_acc, d_cnt,
                                                                      static_cast<unsigned long long*>(ctx->total.p), k, d, sc);
            CU_TRY(cudaGetLastError());
        }
    }
    scan::counts_to_float_kernel<<<(k + 127) / 128, 128, 0, ctx->stream>>>(static_cast<const unsigned long long*>(ctx->total.p), static_cast<float*>(ctx->tcounts.p), k);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(centroids, ctx->cen.p, sizeof(float) * kd, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaMemcpyAsync(total_counts, ctx->tcounts.p, sizeof(float) * k, cudaMemcpyDeviceToHost, ctx->stream));
    if (last_labels && N > 0) CU_TRY(cudaMemcpyAsync(last_labels, ctx->labels.p, sizeof(int) * N, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

int ganrev_assign_cosine_min(ganrev_ctx* ctx, const float* centroids, int k, int32_t* cluster, float* cosv) {
    if (!ctx || !centroids || k < 1) return ctx ? fail(ctx, GANREV_EINVAL, "bad assign arguments") : GANREV_EINVAL;
    if (!ctx->db_ptr) return fail(ctx, GANREV_ESTATE, "database not set");
    CU_TRY(cudaSetDevice(ctx->device));
    const int d = ctx->db_d;
    const int64_t N = ctx->db_n;
    const size_t kd = static_cast<size_t>(k) * d;
    RC_TRY(ensure(ctx, ctx->q, sizeof(float) * kd));
    RC_TRY(ensure(ctx, ctx->rq, sizeof(float) * k));
    RC_TRY(ensure(ctx, ctx->labels, sizeof(int) * static_cast<size_t>(std::max<int64_t>(N, 1))));
    RC_TRY(ensure(ctx, ctx->cosv, sizeof(float) * static_cast<size_t>(std::max<int64_t>(N, 1))));
    CU_TRY(cudaMemcpyAsync(ctx->q.p, centroids, sizeof(float) * kd, cudaMemcpyHostToDevice, ctx->stream));
    RC_TRY(vec_prep(ctx, static_cast<const float*>(ctx->q.p), k, d, static_cast<float*>(ctx->rq.p), nullptr, nullptr));
    scan::ScanParams p{};
    p.db = ctx->db_ptr; p.rdb = static_cast<const float*>(ctx->rdb.p); p.n_rows = N; p.d = d;
    p.q = static_cast<const float*>(ctx->q.p); p.rq = static_cast<const float*>(ctx->rq.p); p.nq = k;
    p.labels = static_cast<int*>(ctx->labels.p); p.cosv = static_cast<float*>(ctx->cosv.p);
    {
        ProfScope ps(ctx, "assign_cosine_min", 2.0 * N * k * d, 4.0 * N * d + 8.0 * N + 4.0 * kd);
        scan::StreamParams sp{};
        size_t smem = 0;
        int grid = 0;
        tfs::TfsParams tp{};
        if (tfs_plan(ctx, p, 2, 0, tp, smem, grid)) RC_TRY((launch_tfs<2, 1>(ctx, tp, smem, grid)));
        else if (label_tc_ok(ctx, p, 2)) RC_TRY((launch_label_tc<2>(ctx, p)));
        else if (rtile_plan(ctx, p, stream_nq(k), 2, sp, smem, grid)) RC_TRY((dispatch_rtile<2>(ctx, stream_nq(k), sp, smem, grid)));
        else if (stream_plan(ctx, p, stream_nq(k), 2, 0, sp, smem, grid)) RC_TRY((dispatch_stream<2, 1>(ctx, stream_nq(k), sp, smem, grid)));
        else if (k <= 16) RC_TRY((launch_assign<1, 2>(ctx, p)));
        else RC_TRY((launch_assign<4, 2>(ctx, p)));
    }
    ctx->assigned = true; ctx->assigned_k = k;
    if (cluster && N > 0) CU_TRY(cudaMemcpyAsync(cluster, ctx->labels.p, sizeof(int) * N, cudaMemcpyDeviceToHost, ctx->stream));
    if (cosv && N > 0) CU_TRY(cudaMemcpyAsync(cosv, ctx->cosv.p, sizeof(float) * N, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

int ganrev_cluster_members(ganrev_ctx* ctx, int k, int m, const float* images, int px, int64_t* member_ids, int32_t* member_counts, float* mean_images) {
    if (!ctx || k < 1 || m < 1 || m > 128 || !member_ids || !member_counts) return ctx ? fail(ctx, GANREV_EINVAL, "bad cluster_members arguments (m must be 1..128)") : GANREV_EINVAL;
    if (!ctx->assigned || ctx->assigned_k != k) return fail(ctx, GANREV_ESTATE, "call ganrev_assign_cosine_min with k=%d first", k);
    CU_TRY(cudaSetDevice(ctx->device));
    const int64_t N = ctx->db_n;
    const bool multi = ctx->world > 1;
    const size_t km = static_cast<size_t>(k) * m;
    RC_TRY(ensure(ctx, ctx->mids, sizeof(long long) * km));
    RC_TRY(ensure(ctx, ctx->mcnt, sizeof(int) * k));
    if (multi) {
        RC_TRY(ensure(ctx, ctx->keys, sizeof(unsigned long long) * (km + k)));                     // local keys, then the unclipped counts
        RC_TRY(ensure(ctx, ctx->keys_all, sizeof(unsigned long long) * km * ctx->world));
        RC_TRY(ensure(ctx, ctx->scores, sizeof(float) * km));
    }
    unsigned long long* d_keys = multi ? static_cast<unsigned long long*>(ctx->keys.p) : nullptr;
    unsigned long long* d_raw = multi ? d_keys + km : nullptr;
    {
        ProfScope ps(ctx, "cluster_members", 0.0, 8.0 * N * k);
        scan::cluster_members_kernel<<<k, 32, 0, ctx->stream>>>(static_cast<const int*>(ctx->labels.p), static_cast<const float*>(ctx->cosv.p), N, m, ctx->db_offset,
                                                               static_cast<long long*>(ctx->mids.p), static_cast<int*>(ctx->mcnt.p), d_keys, d_raw);
        CU_TRY(cudaGetLastError());
    }
    if (multi) {
        // per-cluster top-m across the row shards = the search merge with Q = k clusters (SURVEY 8e): one allgather of the
        // local (cos, global id) keys, one allreduce of the member counts
        NCCL_TRY(ctx->nccl.AllGather(d_keys, ctx->keys_all.p, km, ncclUint64, ctx->comm, ctx->stream));
        NCCL_TRY(ctx->nccl.AllReduce(d_raw, d_raw, k, ncclUint64, ncclSum, ctx->comm, ctx->stream));
        ProfScope ps(ctx, "cluster_members_merge", 0.0, 8.0 * ctx->world * km);
        const unsigned mblocks = static_cast<unsigned>((static_cast<long long>(k) * 32 + scan::kThreads - 1) / scan::kThreads);
        scan::merge_kernel<4><<<mblocks, scan::kThreads, 0, ctx->stream>>>(static_cast<const unsigned long long*>(ctx->keys_all.p), ctx->world, k, m, 0, 0,
            static_cast<long long*>(ctx->mids.p), static_cast<float*>(ctx->scores.p), nullptr);
        scan::cluster_keep_kernel<<<(k + 127) / 128, 128, 0, ctx->stream>>>(d_raw, k, m, static_cast<int*>(ctx->mcnt.p));
        ctx->launches++;
        CU_TRY(cudaGetLastError());
    }
    if (mean_images) {
        if (px < 1) return fail(ctx, GANREV_EINVAL, "px must be positive");
        const float* d_img = nullptr;
        if (images) {
            RC_TRY(ensure(ctx, ctx->stage_a, sizeof(float) * static_cast<size_t>(std::max<int64_t>(N, 1)) * px));
            CU_TRY(cudaMemcpyAsync(ctx->stage_a.p, images, sizeof(float) * static_cast<size_t>(N) * px, cudaMemcpyHostToDevice, ctx->stream));
            d_img = static_cast<const float*>(ctx->stage_a.p);
        } else {
            if (ctx->buf_rows[GANREV_BUF_IMAGES] < N || buf_row_bytes(ctx, GANREV_BUF_IMAGES) != sizeof(float) * static_cast<size_t>(px))
                return fail(ctx, GANREV_ESTATE, "resident IMAGES does not hold %lld x %d", (long long)N, px);
            d_img = static_cast<const float*>(ctx->buf[GANREV_BUF_IMAGES].p);
        }
        RC_TRY(ensure(ctx, ctx->mmean, sizeof(float) * static_cast<size_t>(k) * px));
        if (!multi) {
            ProfScope ps(ctx, "cluster_mean", 1.0 * k * m * px, 4.0 * k * m * px);
            dim3 grid((px + 255) / 256, k);
            scan::cluster_mean_kernel<<<grid, 256, 0, ctx->stream>>>(d_img, px, static_cast<const long long*>(ctx->mids.p), static_cast<const int*>(ctx->mcnt.p), m,
                                                                    static_cast<float*>(ctx->mmean.p));
            CU_TRY(cudaGetLastError());
        } else {
            // the kept images live on whichever rank owns their rows: stage them (a bounded number of clusters at a time),
            // assemble with one integer max-allreduce (every slot has one owner, the others hold zero bits), average in member order
            const int jstep = static_cast<int>(std::max<size_t>(1, std::min<size_t>(k, (size_t(64) << 20) / (static_cast<size_t>(m) * px * 4))));
            RC_TRY(ensure(ctx, ctx->stage_b, sizeof(float) * static_cast<size_t>(jstep) * m * px));
            for (int j0 = 0; j0 < k; j0 += jstep) {
                const int nj = std::min(jstep, k - j0);
                const long long tot = static_cast<long long>(nj) * m * px;
                ProfScope ps(ctx, "cluster_mean", 1.0 * nj * m * px, 8.0 * nj * m * px);
                scan::cluster_stage_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, ctx->stream>>>(d_img, N, ctx->db_offset, px,
                    static_cast<const long long*>(ctx->mids.p), m, j0, nj, static_cast<float*>(ctx->stage_b.p));
                NCCL_TRY(ctx->nccl.AllReduce(ctx->stage_b.p, ctx->stage_b.p, static_cast<size_t>(tot), ncclUint32, ncclMax, ctx->comm, ctx->stream));
                dim3 grid((px + 255) / 256, nj);
                scan::cluster_mean_staged_kernel<<<grid, 256, 0, ctx->stream>>>(static_cast<const float*>(ctx->stage_b.p), px, static_cast<const int*>(ctx->mcnt.p), m, j0,
                                                                               static_cast<float*>(ctx->mmean.p));
                ctx->launches++;
                CU_TRY(cudaGetLastError());
            }
        }
        CU_TRY(cudaMemcpyAsync(mean_images, ctx->mmean.p, sizeof(float) * static_cast<size_t>(k) * px, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU_TRY(cudaMemcpyAsync(member_ids, ctx->mids.p, sizeof(long long) * km, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaMemcpyAsync(member_counts, ctx->mcnt.p, sizeof(int) * k, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

// ---------------------------------------------------------------- measurement hooks
void* ganrev_stream(ganrev_ctx* ctx) { return ctx ? static_cast<void*>(ctx->stream) : nullptr; }
// ---------------------------------------------------------------- R training step (train.cuh; train_r.lua:138-170)
static size_t train_mask_bytes(const TrainR& T, int B) {
    const size_t HW = static_cast<size_t>(T.H) * T.W;
    return (T.fixer ? static_cast<size_t>(B) * T.C * HW : 0) + 2 * static_cast<size_t>(B) * 64 * HW + static_cast<size_t>(B) * 64 * HW / 4 +
           2 * static_cast<size_t>(B) * 128 * HW / 4 + static_cast<size_t>(B) * 128 + static_cast<size_t>(B) * 512;
}
int ganrev_train_R_init(ganrev_ctx* ctx, int C, int H, int W, int noise_dim, int tanh_out, int fixer, const float* blob, size_t n_floats) {
    if (!ctx || !blob) return ctx ? fail(ctx, GANREV_EINVAL, "bad train_R_init arguments") : GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(check_geom(ctx, C, H, W, noise_dim));
    if (ctx->gC != 0 && (ctx->gC != C || ctx->gH != H || ctx->gW != W || ctx->gnd != noise_dim))
        return fail(ctx, GANREV_EINVAL, "the context holds models of another geometry (%dx%dx%d, nd %d)", ctx->gC, ctx->gH, ctx->gW, ctx->gnd);
    TrainR& T = ctx->train;
    T.ready = false;
    T.C = C; T.H = H; T.W = W; T.nd = noise_dim; T.tanh_out = tanh_out ? 1 : 0; T.fixer = fixer ? 1 : 0;
    const int chans[7] = {C, 64, 64, 64, 128, 128, 128};
    size_t o = 0;
    std::vector<unsigned char> flags;
    auto take = [&](size_t n, bool param) { const size_t at = o; o += n; flags.insert(flags.end(), n, param ? 1 : 0); return at; };
    for (int i = 0; i < 6; ++i) {
        T.ci[i] = chans[i]; T.co[i] = chans[i + 1];
        T.cw[i] = take(static_cast<size_t>(T.co[i]) * T.ci[i] * 9, true); T.cb[i] = take(T.co[i], true);
        T.cg[i] = take(T.co[i], true); T.cbe[i] = take(T.co[i], true); T.crm[i] = take(T.co[i], false); T.crv[i] = take(T.co[i], false);
    }
    const size_t F = static_cast<size_t>(128) * (H / 4) * (W / 4);
    T.l1w = take(512 * F, true); T.l1b = take(512, true); T.l1g = take(512, true); T.l1be = take(512, true); T.l1rm = take(512, false); T.l1rv = take(512, false);
    T.l2w = take(static_cast<size_t>(noise_dim) * 512, true); T.l2b = take(noise_dim, true);
    if (o != n_floats) return fail(ctx, GANREV_EINVAL, "R blob has %zu floats, this geometry needs %zu", n_floats, o);
    T.n_floats = o;
    for (DevBuf* b : {&T.P, &T.Gd, &T.M, &T.V}) RC_TRY(ensure(ctx, *b, sizeof(float) * o));
    RC_TRY(ensure(ctx, T.flags, o));
    RC_TRY(ensure(ctx, T.partial, sizeof(double) * 2 * 256));
    RC_TRY(ensure(ctx, T.lossbuf, sizeof(double) * 4));
    CU_TRY(cudaMemcpyAsync(T.P.p, blob, sizeof(float) * o, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemcpyAsync(T.flags.p, flags.data(), o, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaMemsetAsync(T.Gd.p, 0, sizeof(float) * o, ctx->stream));
    CU_TRY(cudaMemsetAsync(T.M.p, 0, sizeof(float) * o, ctx->stream));
    CU_TRY(cudaMemsetAsync(T.V.p, 0, sizeof(float) * o, ctx->stream));
    T.t = 0;
    RC_TRY(finish(ctx));
    T.ready = true;
    return GANREV_OK;
}

int ganrev_train_R_step(ganrev_ctx* ctx, const float* noise, int B, const uint8_t* masks, size_t mask_bytes, const float* hyper7, double* loss2) {
    if (!ctx || !noise || !masks || !hyper7 || B < 2 || B > 1024) return ctx ? fail(ctx, GANREV_EINVAL, "bad train_R_step arguments (2 <= B <= 1024)") : GANREV_EINVAL;
    TrainR& T = ctx->train;
    if (!T.ready) return fail(ctx, GANREV_ESTATE, "call ganrev_train_R_init first");
    if (!ctx->G.loaded) return fail(ctx, GANREV_ESTATE, "G not loaded (the batch is generated by G, train_r.lua:140-141)");
    if (mask_bytes != train_mask_bytes(T, B)) return fail(ctx, GANREV_EINVAL, "masks: %zu bytes given, batch of %d needs %zu", mask_bytes, B, train_mask_bytes(T, B));
    CU_TRY(cudaSetDevice(ctx->device));
    const int C = T.C, H = T.H, W = T.W, nd = T.nd;
    const long long HW = static_cast<long long>(H) * W, HW2 = HW / 4, HW4 = HW / 16;
    const long long F = 128 * HW4;
    // ---- batch: G(noise) in eval mode through the inference kernels
    RC_TRY(stage_input(ctx, GANREV_BUF_NOISE, noise, B));
    RC_TRY(buf_reserve(ctx, GANREV_BUF_IMAGES, B));
    RC_TRY(forward_G_dev(ctx, static_cast<const float*>(ctx->buf[GANREV_BUF_NOISE].p), B, static_cast<float*>(ctx->buf[GANREV_BUF_IMAGES].p)));
    ctx->buf_rows[GANREV_BUF_IMAGES] = B;
    const float* images = static_cast<const float*>(ctx->buf[GANREV_BUF_IMAGES].p);
    const float* d_noise = static_cast<const float*>(ctx->buf[GANREV_BUF_NOISE].p);
    RC_TRY(ensure(ctx, T.masks, mask_bytes));
    CU_TRY(cudaMemcpyAsync(T.masks.p, masks, mask_bytes, cudaMemcpyHostToDevice, ctx->stream));
    const uint8_t* mk = static_cast<const uint8_t*>(T.masks.p);
    const uint8_t* m0 = nullptr;
    if (T.fixer) { m0 = mk; mk += static_cast<size_t>(B) * C * HW; }
    const uint8_t* md[7];
    md[0] = mk; mk += static_cast<size_t>(B) * 64 * HW;  md[1] = mk; mk += static_cast<size_t>(B) * 64 * HW;  md[2] = mk; mk += static_cast<size_t>(B) * 64 * HW2;
    md[3] = mk; mk += static_cast<size_t>(B) * 128 * HW2; md[4] = mk; mk += static_cast<size_t>(B) * 128 * HW2; md[5] = mk; mk += static_cast<size_t>(B) * 128; md[6] = mk;
    // ---- work space: per layer z (conv output), a (ELU output), in (layer input); pooled tensors; statistics; two gradient buffers
    const long long res[6] = {HW, HW, HW, HW2, HW2, HW2};
    size_t need = 0;
    auto carve = [&](size_t n) { const size_t at = need; need += (n + 63) / 64 * 64; return at; };
    size_t oz[6], oa[6], oin[6], omean[7], oistd[7];
    for (int i = 0; i < 6; ++i) { oin[i] = carve(static_cast<size_t>(B) * T.ci[i] * res[i]); oz[i] = carve(static_cast<size_t>(B) * T.co[i] * res[i]); oa[i] = carve(static_cast<size_t>(B) * T.co[i] * res[i]); omean[i] = carve(T.co[i]); oistd[i] = carve(T.co[i]); }
    omean[6] = carve(512); oistd[6] = carve(512);
    const size_t op3 = carve(static_cast<size_t>(B) * 64 * HW2), os6 = carve(static_cast<size_t>(B) * 128 * HW2), op6 = carve(static_cast<size_t>(B) * F);
    const size_t oz7 = carve(static_cast<size_t>(B) * 512), oa7 = carve(static_cast<size_t>(B) * 512), oo7 = carve(static_cast<size_t>(B) * 512), opred = carve(static_cast<size_t>(B) * nd), odpred = carve(static_cast<size_t>(B) * nd);
    const size_t big = static_cast<size_t>(B) * 128 * HW;       // >= every activation
    const size_t og0 = carve(big), og1 = carve(big), og2 = carve(big);
    constexpr int kWgSlices = 8;
    const size_t owg = carve(static_cast<size_t>(kWgSlices) * 128 * 128 * 9);
    const size_t oarg3 = carve((static_cast<size_t>(B) * 64 * HW2 + 3) / 4), oarg6 = carve((static_cast<size_t>(B) * F + 3) / 4);
    RC_TRY(ensure(ctx, T.work, sizeof(float) * need));
    float* wk = static_cast<float*>(T.work.p);
    float* Pp = static_cast<float*>(T.P.p);
    float* Gp = static_cast<float*>(T.Gd.p);
    uint8_t* arg3 = reinterpret_cast<uint8_t*>(wk + oarg3);
    uint8_t* arg6 = reinterpret_cast<uint8_t*>(wk + oarg6);
    auto nb = [](long long n) { return static_cast<unsigned>((n + 255) / 256); };
    // per-channel reductions: one block per channel, as many threads as the channel has 16-byte quads (256 .. 1024)
    auto red_threads = [](long long per_channel) { return static_cast<unsigned>(std::min<long long>(trn::kRedThreads, std::max<long long>(256, (per_channel / 4 + 31) / 32 * 32))); };
    cudaStream_t st = ctx->stream;
    ProfScope ps(ctx, "train_R_step", 6.0 * B * 174.7e6 * (HW / 1024.0), 0.0);
    // ---- forward (training mode)
    if (T.fixer) trn::mask_mul_kernel<<<nb(B * C * HW), 256, 0, st>>>(images, m0, wk + oin[0], B * C * HW);
    else CU_TRY(cudaMemcpyAsync(wk + oin[0], images, sizeof(float) * B * C * HW, cudaMemcpyDeviceToDevice, st));
    for (int i = 0; i < 6; ++i) {
        const int ci = T.ci[i], co = T.co[i], h = i < 3 ? H : H / 2, w = i < 3 ? W : W / 2;
        const long long hw = res[i], tot = static_cast<long long>(B) * co * hw;
        {
            // a thread per 4 pixels of a row; 128 threads = 512 pixels of one image, or several whole images of the small layers
            const unsigned ipb = static_cast<unsigned>(std::max<long long>(1, 128 / (hw / 4)));
            trn::conv3x3_kernel<false><<<dim3(static_cast<unsigned>(ipb > 1 ? 1 : (hw / 4 + 127) / 128), (co + 7) / 8, (B + ipb - 1) / ipb), 128, 8 * ci * 9 * sizeof(float), st>>>(wk + oin[i], Pp + T.cw[i], Pp + T.cb[i], wk + oz[i], B, ci, co, h, w);
        }
        trn::bn_stats_kernel<<<co, red_threads(B * hw), 0, st>>>(wk + oz[i], wk + omean[i], wk + oistd[i], Pp + T.crm[i], Pp + T.crv[i], B, co, static_cast<int>(hw));
        if (i == 2) {          // conv3: ELU -> MaxPool -> Dropout
            trn::bn_elu_drop_kernel<<<nb(tot), 256, 0, st>>>(wk + oz[i], wk + omean[i], wk + oistd[i], Pp + T.cg[i], Pp + T.cbe[i], nullptr, 0, 1.0f, wk + oa[i], nullptr, tot, co, static_cast<int>(hw));
            trn::maxpool_fwd_kernel<<<nb(tot / 4), 256, 0, st>>>(wk + oa[i], wk + op3, arg3, tot / 4, h, w);
            trn::drop_kernel<<<nb(tot / 4), 256, 0, st>>>(wk + op3, md[2], 2.0f, wk + oin[3], tot / 4);
        } else if (i == 5) {   // conv6: ELU -> SpatialDropout -> MaxPool
            trn::bn_elu_drop_kernel<<<nb(tot), 256, 0, st>>>(wk + oz[i], wk + omean[i], wk + oistd[i], Pp + T.cg[i], Pp + T.cbe[i], md[5], 1, 1.0f, wk + oa[i], wk + os6, tot, co, static_cast<int>(hw));
            trn::maxpool_fwd_kernel<<<nb(tot / 4), 256, 0, st>>>(wk + os6, wk + op6, arg6, tot / 4, h, w);
        } else {
            trn::bn_elu_drop_kernel<<<nb(tot), 256, 0, st>>>(wk + oz[i], wk + omean[i], wk + oistd[i], Pp + T.cg[i], Pp + T.cbe[i], md[i], 0, 2.0f, wk + oa[i], wk + oin[i + 1], tot, co, static_cast<int>(hw));
        }
    }
    trn::linear_fwd_kernel<<<nb(static_cast<long long>(B) * 512 * 32), 256, 0, st>>>(wk + op6, Pp + T.l1w, Pp + T.l1b, wk + oz7, B, static_cast<int>(F), 512);
    trn::bn_stats_kernel<<<512, red_threads(B), 0, st>>>(wk + oz7, wk + omean[6], wk + oistd[6], Pp + T.l1rm, Pp + T.l1rv, B, 512, 1);
    trn::bn_elu_drop_kernel<<<nb(B * 512), 256, 0, st>>>(wk + oz7, wk + omean[6], wk + oistd[6], Pp + T.l1g, Pp + T.l1be, md[6], 0, 2.0f, wk + oa7, wk + oo7, B * 512, 512, 1);
    trn::linear_fwd_kernel<<<nb(static_cast<long long>(B) * nd * 32), 256, 0, st>>>(wk + oo7, Pp + T.l2w, Pp + T.l2b, wk + opred, B, 512, nd);
    if (T.tanh_out) trn::tanh_fwd_kernel<<<nb(B * nd), 256, 0, st>>>(wk + opred, B * nd);
    double* lossd = static_cast<double*>(T.lossbuf.p);
    trn::mse_kernel<<<1, 256, 0, st>>>(wk + opred, d_noise, wk + odpred, lossd, B * nd, T.tanh_out);
    CU_TRY(cudaGetLastError());
    // ---- backward
    trn::linear_bwd_w_kernel<<<nb(static_cast<long long>(nd) * 512), 256, 0, st>>>(wk + odpred, wk + oo7, Gp + T.l2w, Gp + T.l2b, B, 512, nd);
    trn::linear_bwd_data_kernel<<<dim3((512 + trn::kLbK - 1) / trn::kLbK, (B + trn::kLbB - 1) / trn::kLbB), trn::kLbK * trn::kLbS, 0, st>>>(wk + odpred, Pp + T.l2w, wk + og0, B, 512, nd);
    trn::drop_elu_bwd_kernel<<<nb(B * 512), 256, 0, st>>>(wk + og0, wk + oa7, md[6], 0, 2.0f, wk + og1, B * 512, 1);
    trn::bn_bwd_reduce_kernel<<<512, red_threads(B), 0, st>>>(wk + og1, wk + oz7, wk + omean[6], wk + oistd[6], Gp + T.l1g, Gp + T.l1be, B, 512, 1);
    trn::bn_bwd_apply_kernel<<<nb(B * 512), 256, 0, st>>>(wk + og1, wk + oz7, wk + omean[6], wk + oistd[6], Pp + T.l1g, Gp + T.l1g, Gp + T.l1be, wk + og0, B * 512, 512, 1, 1.0f / B);
    trn::linear_bwd_w_kernel<<<nb(512 * F), 256, 0, st>>>(wk + og0, wk + op6, Gp + T.l1w, Gp + T.l1b, B, static_cast<int>(F), 512);
    trn::linear_bwd_data_kernel<<<dim3(static_cast<unsigned>((F + trn::kLbK - 1) / trn::kLbK), (B + trn::kLbB - 1) / trn::kLbB), trn::kLbK * trn::kLbS, 0, st>>>(wk + og0, Pp + T.l1w, wk + og1, B, static_cast<int>(F), 512);   // d p6
    float* gcur = wk + og1;     // gradient w.r.t. the OUTPUT of layer i's block (what the next layer consumed)
    float* gA = wk + og0;
    float* gB = wk + og2;
    for (int i = 5; i >= 0; --i) {
        const int ci = T.ci[i], co = T.co[i], h = i < 3 ? H : H / 2, w = i < 3 ? W : W / 2;
        const long long hw = res[i], tot = static_cast<long long>(B) * co * hw;
        // gcur -> gradient w.r.t. the ELU output's consumers, then through dropout / pooling and the ELU: gA = dz
        if (i == 5) {
            trn::maxpool_bwd_kernel<<<nb(tot / 4), 256, 0, st>>>(gcur, arg6, gB, tot / 4, h, w);                 // d s6
            trn::drop_elu_bwd_kernel<<<nb(tot), 256, 0, st>>>(gB, wk + oa[i], md[5], 1, 1.0f, gA, tot, static_cast<int>(hw));
        } else if (i == 2) {
            trn::drop_kernel<<<nb(tot / 4), 256, 0, st>>>(gcur, md[2], 2.0f, gA, tot / 4);                       // d p3
            trn::maxpool_bwd_kernel<<<nb(tot / 4), 256, 0, st>>>(gA, arg3, gB, tot / 4, h, w);                   // d a3
            trn::drop_elu_bwd_kernel<<<nb(tot), 256, 0, st>>>(gB, wk + oa[i], nullptr, 0, 1.0f, gA, tot, static_cast<int>(hw));
        } else {
            trn::drop_elu_bwd_kernel<<<nb(tot), 256, 0, st>>>(gcur, wk + oa[i], md[i], 0, 2.0f, gA, tot, static_cast<int>(hw));
        }
        trn::bn_bwd_reduce_kernel<<<co, red_threads(B * hw), 0, st>>>(gA, wk + oz[i], wk + omean[i], wk + oistd[i], Gp + T.cg[i], Gp + T.cbe[i], B, co, static_cast<int>(hw));
        trn::bn_bwd_apply_kernel<<<nb(tot), 256, 0, st>>>(gA, wk + oz[i], wk + omean[i], wk + oistd[i], Pp + T.cg[i], Gp + T.cg[i], Gp + T.cbe[i], gB, tot, co, static_cast<int>(hw), 1.0f / static_cast<float>(B * hw));   // d conv output
        {
            const int nw = co * ci * 9;
            {   // two cp.async stages exceed the 48 KB default of dynamic shared memory
                static size_t wg_attr_dev[kMaxDevices] = {};
                const size_t need_smem = trn::wgrad_smem_bytes(h, w);
                if (need_smem > wg_attr_dev[ctx->device]) {
                    CU_TRY(cudaFuncSetAttribute(trn::conv3x3_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(need_smem)));
                    wg_attr_dev[ctx->device] = need_smem;
                }
            }
            trn::conv3x3_wgrad_kernel<<<dim3((co + trn::kWgO - 1) / trn::kWgO, (ci + trn::kWgI - 1) / trn::kWgI, kWgSlices), 256, trn::wgrad_smem_bytes(h, w), st>>>(wk + oin[i], gB, wk + owg, B, ci, co, h, w);
            trn::wgrad_sum_kernel<<<nb(nw), 256, 0, st>>>(wk + owg, Gp + T.cw[i], nw, kWgSlices);
        }
        trn::channel_sum_kernel<<<co, red_threads(B * hw), 0, st>>>(gB, Gp + T.cb[i], B, co, static_cast<int>(hw));
        if (i > 0) {
            const unsigned ipb = static_cast<unsigned>(std::max<long long>(1, 128 / (hw / 4)));
            trn::conv3x3_kernel<true><<<dim3(static_cast<unsigned>(ipb > 1 ? 1 : (hw / 4 + 127) / 128), (ci + 7) / 8, (B + ipb - 1) / ipb), 128, 8 * co * 9 * sizeof(float), st>>>(gB, Pp + T.cw[i], nullptr, gA, B, co, ci, h, w);   // d layer input
            float* t = gcur; gcur = gA; gA = t;
        }
    }
    CU_TRY(cudaGetLastError());
    // ---- penalties, clamp, Adam (train_r.lua:150-166; optim.adam)
    trn::penalty_kernel<<<256, 256, 0, st>>>(Pp, static_cast<const uint8_t*>(T.flags.p), static_cast<long long>(T.n_floats), static_cast<double*>(T.partial.p));
    T.t += 1;
    trn::AdamHyper hy{};
    hy.lr = hyper7[0]; hy.beta1 = hyper7[1]; hy.beta2 = hyper7[2]; hy.eps = hyper7[3]; hy.l1 = hyper7[4]; hy.l2 = hyper7[5]; hy.clamp = hyper7[6];
    hy.step_size = static_cast<float>(static_cast<double>(hy.lr) * std::sqrt(1.0 - std::pow(static_cast<double>(hy.beta2), static_cast<double>(T.t))) /
                                      (1.0 - std::pow(static_cast<double>(hy.beta1), static_cast<double>(T.t))));
    trn::adam_kernel<<<nb(static_cast<long long>(T.n_floats)), 256, 0, st>>>(Pp, Gp, static_cast<float*>(T.M.p), static_cast<float*>(T.V.p), static_cast<const uint8_t*>(T.flags.p), static_cast<long long>(T.n_floats), hy);
    CU_TRY(cudaGetLastError());
    ctx->launches += 90;
    double hl[1];
    std::vector<double> part(512);
    CU_TRY(cudaMemcpyAsync(hl, lossd, sizeof(double), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(part.data(), T.partial.p, sizeof(double) * 512, cudaMemcpyDeviceToHost, st));
    RC_TRY(finish(ctx));
    if (loss2) {
        double a = 0.0, q = 0.0;
        for (int k = 0; k < 256; ++k) { a += part[2 * k]; q += part[2 * k + 1]; }
        loss2[0] = hl[0];
        loss2[1] = hl[0] + static_cast<double>(hy.l1) * a + static_cast<double>(hy.l2) * q / 2.0;
    }
    return GANREV_OK;
}

int ganrev_train_R_state(ganrev_ctx* ctx, int what, float* out, size_t n_floats) {
    if (!ctx || !out || what < 0 || what > 3) return ctx ? fail(ctx, GANREV_EINVAL, "bad train_R_state arguments") : GANREV_EINVAL;
    TrainR& T = ctx->train;
    if (!T.ready) return fail(ctx, GANREV_ESTATE, "call ganrev_train_R_init first");
    if (n_floats != T.n_floats) return fail(ctx, GANREV_EINVAL, "state has %zu floats", T.n_floats);
    CU_TRY(cudaSetDevice(ctx->device));
    const DevBuf& b = what == 0 ? T.P : (what == 1 ? T.Gd : (what == 2 ? T.M : T.V));
    CU_TRY(cudaMemcpyAsync(out, b.p, sizeof(float) * n_floats, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

int ganrev_sync(ganrev_ctx* ctx) {
    if (!ctx) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    return finish(ctx);
}
uint64_t ganrev_launch_count(const ganrev_ctx* ctx) { return ctx ? ctx->launches : 0; }
int ganrev_profile_enable(ganrev_ctx* ctx, int on) {
    if (!ctx) return GANREV_EINVAL;
    ctx->prof_on = on != 0;
    return GANREV_OK;
}
int ganrev_profile_reset(ganrev_ctx* ctx) {
    if (!ctx) return GANREV_EINVAL;
    cudaStreamSynchronize(ctx->stream);
    prof_resolve(ctx);
    ctx->prof.clear(); ctx->prof_idx.clear();
    return GANREV_OK;
}
int ganrev_profile_count(ganrev_ctx* ctx) {
    if (!ctx) return 0;
    cudaStreamSynchronize(ctx->stream);
    prof_resolve(ctx);
    return static_cast<int>(ctx->prof.size());
}
int ganrev_profile_get(ganrev_ctx* ctx, int idx, const char** name, uint64_t* launches, double* total_ms, double* flops, double* bytes) {
    if (!ctx || idx < 0 || idx >= static_cast<int>(ctx->prof.size())) return GANREV_EINVAL;
    const ProfEntry& e = ctx->prof[idx];
    if (name) *name = e.name.c_str();
    if (launches) *launches = e.launches;
    if (total_ms) *total_ms = e.total_ms;
    if (flops) *flops = e.flops;
    if (bytes) *bytes = e.bytes;
    return GANREV_OK;
}
// bench.py --config 5: a synthetic N(0,1) database generated on the device (SURVEY 8d: "generated on device" so that
// no 10 GB host upload is timed); counter-based, so any sharding of the rows gives the same values for the same global row.
int ganrev_debug_db_synthetic(ganrev_ctx* ctx, int64_t N, int d, uint64_t seed, int64_t global_row0) {
    if (!ctx || N < 0 || d < 1) return ctx ? fail(ctx, GANREV_EINVAL, "bad db_synthetic arguments") : GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    ctx->db_ptr = nullptr; ctx->db_n = 0;
    RC_TRY(ensure(ctx, ctx->db, sizeof(float) * static_cast<size_t>(std::max<int64_t>(N, 1)) * d));
    const long long tot = static_cast<long long>(N) * d;
    synthetic_normal_kernel<<<static_cast<unsigned>(std::min<long long>((tot + 255) / 256, 1 << 20)), 256, 0, ctx->stream>>>(
        static_cast<float*>(ctx->db.p), tot, seed, static_cast<unsigned long long>(global_row0) * d);
    ctx->launches++;
    CU_TRY(cudaGetLastError());
    RC_TRY(finish(ctx));
    // adopt it as the database through the normal path (device-to-device "upload" of itself is skipped: db.p already holds it)
    return ganrev_db_adopt_own(ctx, N, d);
}
// The approximate cosines of the tensor-core filter for every (query, row) pair of a SMALL database, so that tests can measure
// |approximate - exact| against the bound eps(d) the filter relies on (search_tc.cuh).  out [Q x N]; eps_out = eps(d).
int ganrev_debug_tc_scores(ganrev_ctx* ctx, const float* queries, int Q, float* out, float* eps_out) {
    if (!ctx || !queries || Q < 1 || !out) return ctx ? fail(ctx, GANREV_EINVAL, "bad tc_scores arguments") : GANREV_EINVAL;
    if (!ctx->db_ptr) return fail(ctx, GANREV_ESTATE, "database not set");
    const int d = ctx->db_d, kp = stc::packed_cols(d);
    const int64_t N = ctx->db_n;
    if (d > 1024 || static_cast<double>(N) * Q > 1.0e8) return fail(ctx, GANREV_EINVAL, "tc_scores is a debug hook for small problems");
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(ensure(ctx, ctx->q, sizeof(float) * static_cast<size_t>(Q) * d));
    RC_TRY(ensure(ctx, ctx->rq, sizeof(float) * Q));
    CU_TRY(cudaMemcpyAsync(ctx->q.p, queries, sizeof(float) * static_cast<size_t>(Q) * d, cudaMemcpyHostToDevice, ctx->stream));
    RC_TRY(vec_prep(ctx, static_cast<const float*>(ctx->q.p), Q, d, static_cast<float*>(ctx->rq.p), nullptr, nullptr));
    RC_TRY(ensure(ctx, ctx->tc_flags, 4 * sizeof(int)));
    CU_TRY(cudaMemsetAsync(ctx->tc_flags.p, 0, 4 * sizeof(int), ctx->stream));
    if (!ctx->pdb_valid) {
        RC_TRY(tc_pack(ctx, "search_tc_pack_db", ctx->db_ptr, static_cast<const float*>(ctx->rdb.p), N, d, ctx->pdb, false));
        ctx->pdb_valid = true;
    }
    RC_TRY(tc_pack(ctx, "search_tc_pack_q", static_cast<const float*>(ctx->q.p), static_cast<const float*>(ctx->rq.p), Q, d, ctx->pq, true));
    RC_TRY(ensure(ctx, ctx->tc_thr, sizeof(float) * Q));
    RC_TRY(ensure(ctx, ctx->tc_cnt, sizeof(unsigned) * (3 * static_cast<size_t>(Q) + 4)));
    RC_TRY(ensure(ctx, ctx->tc_pairs, sizeof(uint4) * 16));
    RC_TRY(ensure(ctx, ctx->tc_dump, sizeof(float) * static_cast<size_t>(Q) * N));
    CU_TRY(cudaMemsetAsync(ctx->tc_thr.p, 0x7f, sizeof(float) * Q, ctx->stream));     // 0x7f7f7f7f = 3.39e38: nothing passes
    CU_TRY(cudaMemsetAsync(ctx->tc_cnt.p, 0, sizeof(unsigned) * (3 * static_cast<size_t>(Q) + 4), ctx->stream));
    CU_TRY(cudaMemsetAsync(ctx->tc_dump.p, 0, sizeof(float) * static_cast<size_t>(Q) * N, ctx->stream));
    CU_TRY(cudaFuncSetAttribute(stc::filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, stc::kSmem));
    CUtensorMap tmQ, tmX;
    RC_TRY(tc_make_map(ctx, &tmQ, ctx->pq.p, kp, Q, kp, stc::QM));
    RC_TRY(tc_make_map(ctx, &tmX, ctx->pdb.p, kp, N, kp, stc::RN));
    stc::FilterParams fp{};
    fp.nq = Q; fp.n_rows = N; fp.stride = 1; fp.d = d; fp.nslices = kp / 128;
    fp.q_tiles = (Q + stc::QM - 1) / stc::QM;
    fp.items = static_cast<long long>(fp.q_tiles) * ((N + stc::RN - 1) / stc::RN);
    fp.thr = static_cast<const float*>(ctx->tc_thr.p); fp.cnt = static_cast<unsigned*>(ctx->tc_cnt.p);
    fp.pairs = static_cast<uint4*>(ctx->tc_pairs.p); fp.total = static_cast<unsigned*>(ctx->tc_cnt.p) + 3 * Q; fp.pair_cap = 0;
    fp.flags = static_cast<int*>(ctx->tc_flags.p) + 3; fp.err_flag = ctx->d_err_flag;
    fp.dump = static_cast<float*>(ctx->tc_dump.p);
    {
        ProfScope ps(ctx, "search_tc_filter_dump", 0.0, 0.0);
        stc::filter_kernel<true><<<static_cast<int>(std::min<long long>(fp.items, ctx->num_sms)), stc::kThr, stc::kSmem, ctx->stream>>>(tmQ, tmX, fp);
        CU_TRY(cudaGetLastError());
    }
    CU_TRY(cudaMemcpyAsync(out, ctx->tc_dump.p, sizeof(float) * static_cast<size_t>(Q) * N, cudaMemcpyDeviceToHost, ctx->stream));
    if (eps_out) *eps_out = stc::tc_eps(d);
    return finish(ctx);
}
// [0] searches answered by the tensor-core path, [1] searches re-run on the fmaf-chain kernels (flags raised)
int ganrev_debug_tc_counters(ganrev_ctx* ctx, uint64_t* out2) {
    if (!ctx || !out2) return GANREV_EINVAL;
    out2[0] = ctx->tc_searches; out2[1] = ctx->tc_fallbacks;
    return GANREV_OK;
}
int ganrev_debug_tfs_stats(ganrev_ctx* ctx, uint64_t* out4) {
    if (!ctx || !out4) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    out4[0] = out4[1] = out4[2] = 0; out4[3] = ctx->tfs_launches;
    ctx->tfs_launches = 0;
    if (ctx->tfs_aux.p) {
        unsigned long long* st = reinterpret_cast<unsigned long long*>(static_cast<unsigned*>(ctx->tfs_aux.p) + 32);
        CU_TRY(cudaMemcpyAsync(out4, st, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaMemsetAsync(st, 0, 4 * sizeof(unsigned long long), ctx->stream));
        return finish(ctx);
    }
    return GANREV_OK;
}
// Measured fp32 FMA throughput of this GPU at its current clocks (the roof the exact fmaf-chain kernels are graded against;
// MEASURED_PEAKS.json has no fp32 figure): 8 independent chains per thread, all SMs, ~50 ms.
int ganrev_debug_fma_peak(ganrev_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(ensure(ctx, ctx->thr, sizeof(double)));
    const int iters = 1 << 16, blocks = ctx->num_sms * 8, threads = 256;
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0)); CU_TRY(cudaEventCreate(&e1));
    fma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(static_cast<float*>(ctx->thr.p), 1024, 1.0f);   // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0, ctx->stream);
        fma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(static_cast<float*>(ctx->thr.p), iters, 1.0f);
        cudaEventRecord(e1, ctx->stream);
        cudaEventSynchronize(e1);
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double fl = 2.0 * 16.0 * iters * static_cast<double>(blocks) * threads;
        best = std::max(best, fl / (ms * 1e-3) * 1e-12);
    }
    ctx->launches += 4;
    double best2 = 0.0;
    fma2_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(static_cast<float*>(ctx->thr.p), 1024, 1.0f);
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0, ctx->stream);
        fma2_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(static_cast<float*>(ctx->thr.p), iters, 1.0f);
        cudaEventRecord(e1, ctx->stream);
        cudaEventSynchronize(e1);
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double fl = 2.0 * 16.0 * iters * static_cast<double>(blocks) * threads;
        best2 = std::max(best2, fl / (ms * 1e-3) * 1e-12);
    }
    ctx->launches += 4;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops = best;
    if (getenv("GANREV_PRINT_FMA2")) fprintf(stderr, "fp32 FFMA %.1f TFLOP/s, FFMA2 (fma.rn.f32x2) %.1f TFLOP/s\n", best, best2);
    return finish(ctx);
}
// Debug: arm a clock64 timeline of CTA 0 for the named tensor-core layer / read it back ([8][256] int64).
int ganrev_debug_trace_arm(ganrev_ctx* ctx, const char* layer) {
    if (!ctx || !layer) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    RC_TRY(ensure(ctx, ctx->trace, 8 * 256 * sizeof(long long)));
    CU_TRY(cudaMemsetAsync(ctx->trace.p, 0, 8 * 256 * sizeof(long long), ctx->stream));
    ctx->trace_layer = layer;
    return finish(ctx);
}
int ganrev_debug_trace_read(ganrev_ctx* ctx, int64_t* out) {
    if (!ctx || !out || !ctx->trace.p) return GANREV_EINVAL;
    CU_TRY(cudaSetDevice(ctx->device));
    CU_TRY(cudaMemcpyAsync(out, ctx->trace.p, 8 * 256 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}
int ganrev_set_option(ganrev_ctx* ctx, const char* name, int64_t value) {
    if (!ctx || !name) return GANREV_EINVAL;
    if (!strcmp(name, "chunk")) {
        if (value < 0 || value > (1 << 20)) return fail(ctx, GANREV_EINVAL, "chunk out of range");   // 0 = automatic
        ctx->chunk = value;
        return GANREV_OK;
    }
    if (!strcmp(name, "rtile")) { ctx->rtile = value != 0; return GANREV_OK; }
    if (!strcmp(name, "search_tc")) { ctx->search_tc = value != 0; return GANREV_OK; }
    if (!strcmp(name, "label_tc")) { ctx->label_tc = value != 0; return GANREV_OK; }
    if (!strcmp(name, "stream_tc")) { ctx->stream_tc = value != 0; return GANREV_OK; }
    if (!strcmp(name, "kmeans_tc")) { ctx->kmeans_tc = value != 0; return GANREV_OK; }
    if (!strcmp(name, "tma_hybrid")) { ctx->tma_hybrid = value != 0; return GANREV_OK; }
    if (!strcmp(name, "ups_cycles")) { ctx->ups_cycles = value < 1 ? 1 : static_cast<int>(value); return GANREV_OK; }
    if (!strcmp(name, "pdl")) { ctx->pdl = value != 0; return GANREV_OK; }
    if (!strcmp(name, "xpose2")) { ctx->xpose2 = value < 0 ? 0 : (value > 2 ? 2 : static_cast<int>(value)); return GANREV_OK; }   // read at load time
    if (!strcmp(name, "fuse_conv3")) { ctx->fuse_conv3 = value < 0 ? 0 : (value > 2 ? 2 : static_cast<int>(value)); return GANREV_OK; }   // read by ganrev_load_G
    if (!strcmp(name, "tma_store")) { ctx->tma_store = value < 0 ? 0 : (value > 2 ? 2 : static_cast<int>(value)); return GANREV_OK; }
    if (!strcmp(name, "conv_impl")) {
        if (value != 0 && value != 1) return fail(ctx, GANREV_EINVAL, "conv_impl must be 0 or 1");
        ctx->conv_impl = static_cast<int>(value);
        return GANREV_OK;
    }
    if (!strcmp(name, "cta_pairs")) { ctx->cta_pairs = static_cast<int>(value); return GANREV_OK; }
    if (!strcmp(name, "dbg")) { ctx->dbg = static_cast<int>(value); return GANREV_OK; }
    return fail(ctx, GANREV_EINVAL, "unknown option %s", name);
}

}  // extern "C"

// layers.cuh -- the shallow / narrow layers that stay on CUDA cores (SURVEY.md section 8a):
//   * noise fp32 -> bf16 K-padded rows (A operand of G's Linear, models.lua:115)
//   * R conv1  C->64, K = 9*C      (models.lua:399-411) fp32 NCHW in (+ explicit dropout
//     mask fused into the loader), folded BN + ELU, bf16 NHWC out
//   * torch.dist over image pairs  (apply_r.lua:366) in the canonical lane-tree order
//   * the 15%-quantile threshold + flags (apply_r.lua:370-378) as a device radix select
#pragma once
#include "common.cuh"

namespace ganrev {

// ------------------------------------------------------------------ noise -> bf16 [n][kpad]
__global__ void noise_to_bf16_kernel(const float* __restrict__ in, int nd, int kpad, bf16* __restrict__ out, long long n) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= n * kpad) return;
    const long long r = idx / kpad;
    const int c = static_cast<int>(idx - r * kpad);
    out[idx] = __float2bfloat16_rn(c < nd ? in[r * nd + c] : 0.0f);
}

// ------------------------------------------------------------------ R conv1
// wsm layout: [k = (ci*3+ky)*3+kx][64] fp32, then scale[64], shift[64].
template <int CIN>
__global__ void __launch_bounds__(128)
r_conv1_kernel(const float* __restrict__ img, const uint8_t* __restrict__ mask, const float* __restrict__ wpack,
               bf16* __restrict__ out, int H, int W, long long npix_total) {
    constexpr int K = CIN * 9;
    __shared__ __align__(16) float wsm[K * 64 + 128];
    for (int i = threadIdx.x; i < K * 64 + 128; i += blockDim.x) wsm[i] = wpack[i];
    __syncthreads();
    const long long pix = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool live = pix < npix_total;          // dead tail threads still take part in the warp store
    const int w = static_cast<int>(pix % W);
    const int h = static_cast<int>((pix / W) % H);
    const long long n = pix / (static_cast<long long>(W) * H);
    float acc[64];
#pragma unroll
    for (int c = 0; c < 64; ++c) acc[c] = 0.0f;
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
        const long long plane = (n * CIN + ci) * static_cast<long long>(H) * W;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int hh = h + ky - 1;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int ww = w + kx - 1;
                float x = 0.0f;
                if (live && hh >= 0 && hh < H && ww >= 0 && ww < W) {
                    const long long off = plane + static_cast<long long>(hh) * W + ww;
                    x = img[off];
                    if (mask != nullptr && mask[off] == 0) x = 0.0f;   // v1 dropout: x*mask, no rescale
                }
                const float4* wr = reinterpret_cast<const float4*>(wsm + ((ci * 3 + ky) * 3 + kx) * 64);
#pragma unroll
                for (int c4 = 0; c4 < 16; ++c4) {
                    const float4 wv = wr[c4];
                    acc[4 * c4 + 0] = fmaf(x, wv.x, acc[4 * c4 + 0]);
                    acc[4 * c4 + 1] = fmaf(x, wv.y, acc[4 * c4 + 1]);
                    acc[4 * c4 + 2] = fmaf(x, wv.z, acc[4 * c4 + 2]);
                    acc[4 * c4 + 3] = fmaf(x, wv.w, acc[4 * c4 + 3]);
                }
            }
        }
    }
    const float* sc = wsm + K * 64;
    const float* sh = sc + 64;
    // A warp's 32 pixels are 4 KB contiguous in the NHWC output: stage through shared memory
    // (16-byte chunks XOR-swizzled by pixel) so the global stores are fully coalesced.
    __shared__ uint4 stage[128 * 8];
    const int lane = threadIdx.x & 31;
    uint4* wstage = stage + (threadIdx.x >> 5) * 256;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = elu_fast(fmaf(acc[8 * j + t], sc[8 * j + t], sh[8 * j + t]));
        uint4 pk;
        __nv_bfloat162 b0 = __floats2bfloat162_rn(v[0], v[1]), b1 = __floats2bfloat162_rn(v[2], v[3]);
        __nv_bfloat162 b2 = __floats2bfloat162_rn(v[4], v[5]), b3 = __floats2bfloat162_rn(v[6], v[7]);
        pk.x = *reinterpret_cast<uint32_t*>(&b0); pk.y = *reinterpret_cast<uint32_t*>(&b1);
        pk.z = *reinterpret_cast<uint32_t*>(&b2); pk.w = *reinterpret_cast<uint32_t*>(&b3);
        wstage[lane * 8 + (j ^ (lane & 7))] = pk;
    }
    __syncwarp();
    const long long warp_pix0 = pix - lane;                       // first pixel of this warp
    uint4* o = reinterpret_cast<uint4*>(out + warp_pix0 * 64);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int e = i * 32 + lane;                              // 16-byte element of the 4 KB block
        const int t = e >> 3, c = e & 7;
        if (warp_pix0 + t < npix_total) o[e] = wstage[t * 8 + (c ^ (t & 7))];
    }
}

// ------------------------------------------------------------------ G conv3, pass 2
// Pass 1 (tensor cores) left P[tap*C + co][n][y][x] = w[co][:, tap] . act[n][y][x][:] (one plane of
// `plane` floats per tap and output channel) for every INPUT pixel; the 3x3 conv output is the sum of the 9 neighbours' matching tap products
// (out-of-image neighbours contribute nothing = zero padding), + bias, then Sigmoid
// (models.lua:132-133).  fp32 NCHW out.  One thread per FOUR consecutive output pixels of a row (W is a power of two >= 16):
// each tap plane is read as one aligned 16-byte load plus, for the left / right taps, one edge float -- 15 loads per 4 pixels
// instead of 36, shifts instead of divisions (the one-pixel version was issue-bound at 2.7 TB/s).  Every pixel still adds its
// taps in (ky, kx) order.
template <int COUT>
__global__ void __launch_bounds__(256)
g_conv3_gather_kernel(const float* __restrict__ P, long long plane, const float* __restrict__ bias, float* __restrict__ out,
                      int H, int W, int lgH, int lgW, long long n_img) {
    const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;     // quad of pixels
    if (q >= ((n_img << (lgH + lgW)) >> 2)) return;
    const long long pix = q << 2;                                                          // (n*H + y)*W + x0
    const int x0 = static_cast<int>(pix) & (W - 1);
    const int y = static_cast<int>(pix >> lgW) & (H - 1);
    const long long n = pix >> (lgH + lgW);
    float acc[COUT][4];
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
        const float b = __ldg(bias + co);
        acc[co][0] = acc[co][1] = acc[co][2] = acc[co][3] = b;
    }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int yy = y + ky - 1;
        if (yy < 0 || yy >= H) continue;
        const long long row = pix + static_cast<long long>(ky - 1) * W;                    // pixel (n, yy, x0)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                const float* pl = P + static_cast<long long>((ky * 3 + kx) * COUT + co) * plane + row;
                const float4 v = __ldg(reinterpret_cast<const float4*>(pl));
                if (kx == 0) {          // output x reads input x - 1
                    if (x0 > 0) acc[co][0] += __ldg(pl - 1);
                    acc[co][1] += v.x; acc[co][2] += v.y; acc[co][3] += v.z;
                } else if (kx == 1) {
                    acc[co][0] += v.x; acc[co][1] += v.y; acc[co][2] += v.z; acc[co][3] += v.w;
                } else {                // output x reads input x + 1
                    acc[co][0] += v.y; acc[co][1] += v.z; acc[co][2] += v.w;
                    if (x0 + 4 < W) acc[co][3] += __ldg(pl + 4);
                }
            }
        }
    }
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
        float4 o;
        o.x = 1.0f / (1.0f + __expf(-acc[co][0])); o.y = 1.0f / (1.0f + __expf(-acc[co][1]));
        o.z = 1.0f / (1.0f + __expf(-acc[co][2])); o.w = 1.0f / (1.0f + __expf(-acc[co][3]));
        *reinterpret_cast<float4*>(out + (((n * COUT + co) << lgH) + y) * static_cast<long long>(W) + x0) = o;
    }
}

// ------------------------------------------------------------------ torch.dist, batched
// Canonical order (mirrored by oracle orc_l2): element i belongs to lane (i/4)%32, each lane
// adds its fp32 squares in ascending i into a double, then an xor-butterfly over the lanes.
// MASKED (the masked refinement's distance, DESIGN.md section 4.7): keep[] is a uint8 [n][px] keep-mask and the difference is
// keep ? x - y : 0 in the same order, so the result is bit-identical to the unmasked kernel on where(keep, x, 0), where(keep, y, 0)
// (a +0 square added to the double sum changes no bit) and the values under keep = 0 never matter, even NaN / Inf.
template <bool MASKED = false>
__global__ void __launch_bounds__(256)
l2_pairs_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n, int px, double* __restrict__ l2,
                const uint8_t* __restrict__ keep) {
    const int lane = threadIdx.x & 31;
    const long long pair = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (pair >= n) return;
    const float* x = a + pair * px;
    const float* y = b + pair * px;
    const uint8_t* k = MASKED ? keep + pair * px : nullptr;
    double s = 0.0;
    bool vec = ((px & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((reinterpret_cast<uintptr_t>(y) & 15) == 0);
    if constexpr (MASKED) vec = vec && ((reinterpret_cast<uintptr_t>(k) & 3) == 0);
    if (vec) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
        const float4* y4 = reinterpret_cast<const float4*>(y);
        const uchar4* k4 = reinterpret_cast<const uchar4*>(k);
        const int n4 = px >> 2;
        int i = lane;
        // 4 independent 128-bit loads per operand in flight
        for (; i + 96 < n4; i += 128) {
            float4 xa[4], ya[4];
            uchar4 ka[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { xa[u] = __ldcs(x4 + i + 32 * u); ya[u] = __ldcs(y4 + i + 32 * u); }
            if constexpr (MASKED) {
#pragma unroll
                for (int u = 0; u < 4; ++u) ka[u] = __ldcs(k4 + i + 32 * u);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float d0 = __fsub_rn(xa[u].x, ya[u].x), d1 = __fsub_rn(xa[u].y, ya[u].y);
                float d2 = __fsub_rn(xa[u].z, ya[u].z), d3 = __fsub_rn(xa[u].w, ya[u].w);
                if constexpr (MASKED) {
                    d0 = ka[u].x != 0 ? d0 : 0.0f; d1 = ka[u].y != 0 ? d1 : 0.0f;
                    d2 = ka[u].z != 0 ? d2 : 0.0f; d3 = ka[u].w != 0 ? d3 : 0.0f;
                }
                s += static_cast<double>(__fmul_rn(d0, d0));
                s += static_cast<double>(__fmul_rn(d1, d1));
                s += static_cast<double>(__fmul_rn(d2, d2));
                s += static_cast<double>(__fmul_rn(d3, d3));
            }
        }
        for (; i < n4; i += 32) {
            const float4 xv = __ldcs(x4 + i), yv = __ldcs(y4 + i);
            float d0 = __fsub_rn(xv.x, yv.x), d1 = __fsub_rn(xv.y, yv.y);
            float d2 = __fsub_rn(xv.z, yv.z), d3 = __fsub_rn(xv.w, yv.w);
            if constexpr (MASKED) {
                const uchar4 kv = __ldcs(k4 + i);
                d0 = kv.x != 0 ? d0 : 0.0f; d1 = kv.y != 0 ? d1 : 0.0f;
                d2 = kv.z != 0 ? d2 : 0.0f; d3 = kv.w != 0 ? d3 : 0.0f;
            }
            s += static_cast<double>(__fmul_rn(d0, d0));
            s += static_cast<double>(__fmul_rn(d1, d1));
            s += static_cast<double>(__fmul_rn(d2, d2));
            s += static_cast<double>(__fmul_rn(d3, d3));
        }
    } else {
        for (int base = lane * 4; base < px; base += 128)
            for (int j = 0; j < 4 && base + j < px; ++j) {
                float d = __fsub_rn(x[base + j], y[base + j]);
                if constexpr (MASKED) d = k[base + j] != 0 ? d : 0.0f;
                s += static_cast<double>(__fmul_rn(d, d));
            }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) l2[pair] = __dsqrt_rn(s);
}

// ------------------------------------------------------------------ nearest set image by torch.dist
// sample.lua:128-148 (findClosestNeighboursOf): for each query image scan the whole training set and
// keep the first strictly smaller torch.dist.  One warp per set row, QB queries per pass: the row's
// 128-float pieces are loaded once and compared against QB query rows (L1/L2 resident), each
// (row, query) distance summed in the canonical lane order of l2_pairs_kernel.  Every warp keeps its
// own best (distance, row) per query -- rows arrive in ascending order inside a warp, so strict <
// keeps the lowest row -- and a second kernel merges the warps by (distance, row) and applies the
// reference's quirk that row 0 is taken unconditionally (a NaN there sticks).
constexpr int NL2_QB = 8;
struct NearestRec { double d; long long id; };

__global__ void __launch_bounds__(256)
nearest_l2_kernel(const float* __restrict__ q, int Q, int q0, const float* __restrict__ set, long long N, int px,
                  NearestRec* __restrict__ partial /* [gridDim.x * 8 warps][NL2_QB] */, unsigned char* __restrict__ row0_nan /* [Q] */) {
    const int lane = threadIdx.x & 31;
    const long long gw = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nw = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    const int nq = min(NL2_QB, Q - q0);
    double bd[NL2_QB];
    long long bi[NL2_QB];
#pragma unroll
    for (int v = 0; v < NL2_QB; ++v) { bd[v] = 0.0; bi[v] = -1; }
    const bool vec = ((px & 3) == 0) && ((reinterpret_cast<uintptr_t>(set) & 15) == 0) && ((reinterpret_cast<uintptr_t>(q) & 15) == 0);
    for (long long row = gw; row < N; row += nw) {
        const float* x = set + row * px;
        double s[NL2_QB];
#pragma unroll
        for (int v = 0; v < NL2_QB; ++v) s[v] = 0.0;
        if (vec) {
            const float4* x4 = reinterpret_cast<const float4*>(x);
            const int n4 = px >> 2;
            for (int i = lane; i < n4; i += 32) {
                const float4 xv = __ldcs(x4 + i);
#pragma unroll
                for (int v = 0; v < NL2_QB; ++v) {
                    if (v < nq) {
                        const float4 yv = __ldg(reinterpret_cast<const float4*>(q + static_cast<long long>(q0 + v) * px) + i);
                        // torch.dist(trainingSet[j], img): set row minus query, squared in fp32, summed in double
                        const float d0 = __fsub_rn(xv.x, yv.x), d1 = __fsub_rn(xv.y, yv.y);
                        const float d2 = __fsub_rn(xv.z, yv.z), d3 = __fsub_rn(xv.w, yv.w);
                        s[v] += static_cast<double>(__fmul_rn(d0, d0));
                        s[v] += static_cast<double>(__fmul_rn(d1, d1));
                        s[v] += static_cast<double>(__fmul_rn(d2, d2));
                        s[v] += static_cast<double>(__fmul_rn(d3, d3));
                    }
                }
            }
        } else {
            for (int base = lane * 4; base < px; base += 128)
                for (int j = 0; j < 4 && base + j < px; ++j) {
                    const float xv = x[base + j];
#pragma unroll
                    for (int v = 0; v < NL2_QB; ++v)
                        if (v < nq) {
                            const float d = __fsub_rn(xv, q[static_cast<long long>(q0 + v) * px + base + j]);
                            s[v] += static_cast<double>(__fmul_rn(d, d));
                        }
                }
        }
#pragma unroll
        for (int v = 0; v < NL2_QB; ++v) {
            double t = s[v];
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) t = t + __shfl_xor_sync(0xffffffffu, t, off);
            const double dist = __dsqrt_rn(t);
            if (v < nq) {
                if (bi[v] < 0 ? !(dist != dist) : dist < bd[v]) { bd[v] = dist; bi[v] = row; }   // NaN never wins here
                if (row == 0 && lane == 0) row0_nan[q0 + v] = (dist != dist) ? 1 : 0;
            }
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int v = 0; v < NL2_QB; ++v) { partial[gw * NL2_QB + v].d = bd[v]; partial[gw * NL2_QB + v].id = bi[v]; }
    }
}

// one warp per query of the pass: min over the per-warp records by (distance, row).  quirk = 1 applies the reference's
// "row 0 is taken unconditionally" rule here (single rank); quirk = 0 leaves it to nearest_l2_ranks_kernel.
__global__ void nearest_l2_merge_kernel(const NearestRec* __restrict__ partial, long long n_warps, int Q, int q0, long long N,
                                        const unsigned char* __restrict__ row0_nan, int quirk, long long* __restrict__ ids, double* __restrict__ dist) {
    const int v = blockIdx.x, lane = threadIdx.x;
    if (q0 + v >= Q) return;
    double bd = 0.0;
    long long bi = -1;
    for (long long w = lane; w < n_warps; w += 32) {
        const NearestRec r = partial[w * NL2_QB + v];
        if (r.id >= 0 && (bi < 0 || r.d < bd || (r.d == bd && r.id < bi))) { bd = r.d; bi = r.id; }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, bd, off);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, off);
        if (oi >= 0 && (bi < 0 || od < bd || (od == bd && oi < bi))) { bd = od; bi = oi; }
    }
    if (lane == 0) {
        if (quirk && N > 0 && (row0_nan[q0 + v] || bi < 0)) {      // row 0 was NaN (it sticks), or every distance was NaN (row 0 again)
            ids[q0 + v] = 0;
            dist[q0 + v] = __longlong_as_double(0x7ff8000000000000ll);
        } else {
            ids[q0 + v] = bi;
            dist[q0 + v] = bi < 0 ? __longlong_as_double(0x7ff0000000000000ll) : bd;   // empty set: -1, +inf
        }
    }
}
// Row-sharded set: rec[r][q] = {distance, global row or -1, row0-was-NaN flag of the rank that owns global row 0}; every rank
// merges the allgathered records identically.
struct NearestRankRec { double d; long long id; long long row0_nan; long long pad; };
__global__ void nearest_l2_pack_kernel(const long long* __restrict__ ids, const double* __restrict__ dist, const unsigned char* __restrict__ row0_nan,
                                       int Q, long long offset, int owns_row0, NearestRankRec* __restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    NearestRankRec r;
    r.d = dist[q]; r.id = ids[q] < 0 ? -1 : ids[q] + offset; r.row0_nan = owns_row0 ? row0_nan[q] : 0; r.pad = 0;
    out[q] = r;
}
__global__ void nearest_l2_ranks_kernel(const NearestRankRec* __restrict__ all, int world, int Q, long long n_total,
                                        long long* __restrict__ ids, double* __restrict__ dist) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    double bd = 0.0;
    long long bi = -1;
    bool stick = false;
    for (int r = 0; r < world; ++r) {
        const NearestRankRec c = all[static_cast<long long>(r) * Q + q];
        stick |= c.row0_nan != 0;
        if (c.id >= 0 && (bi < 0 || c.d < bd || (c.d == bd && c.id < bi))) { bd = c.d; bi = c.id; }
    }
    if (n_total > 0 && (stick || bi < 0)) { ids[q] = 0; dist[q] = __longlong_as_double(0x7ff8000000000000ll); }
    else { ids[q] = bi; dist[q] = bi < 0 ? __longlong_as_double(0x7ff0000000000000ll) : bd; }
}

// ------------------------------------------------------------------ quantile threshold + flags
__device__ __forceinline__ unsigned long long f64_key(double v) {   // ascending order-preserving
    const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double f64_unkey(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    return __longlong_as_double(static_cast<long long>(b));
}
// MSB radix select of the rank-th smallest (0-based) of sims = 1 - l2, 8 bits per pass, any number of blocks and
// (with one 256-bin integer allreduce per pass between the two kernels) any number of ranks: every rank sees the same
// global histogram, so every rank walks the same prefix.  state = {prefix, rank, n_total}, hist = 256 bins (uint64).
__global__ void quantile_init_kernel(unsigned long long* __restrict__ state, unsigned long long* __restrict__ hist, long long rank_or_neg,
                                     double quantile) {
    hist[threadIdx.x] = 0ull;
    if (threadIdx.x == 0) {
        state[0] = 0ull;
        // multi-rank: state[2] holds the allreduced n_calc; rank = floor(n_total * quantile) - 1 (apply_r.lua:371, 1-based index)
        state[1] = rank_or_neg >= 0 ? static_cast<unsigned long long>(rank_or_neg)
                                    : static_cast<unsigned long long>(static_cast<long long>(floor(static_cast<double>(static_cast<long long>(state[2])) * quantile)) - 1);
    }
}
__global__ void __launch_bounds__(256)
quantile_hist_kernel(const double* __restrict__ l2, long long n, const unsigned long long* __restrict__ state, int pass,
                     unsigned long long* __restrict__ hist) {
    __shared__ unsigned int sh[256];
    sh[threadIdx.x] = 0u;
    __syncthreads();
    const int shift = 56 - 8 * pass;
    const unsigned long long prefix = state[0];
    const unsigned long long himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned long long k = f64_key(1.0 - l2[i]);
        if ((k & himask) == prefix) atomicAdd(&sh[(k >> shift) & 0xFF], 1u);
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], static_cast<unsigned long long>(sh[threadIdx.x]));
}
__global__ void quantile_pick_kernel(unsigned long long* __restrict__ state, unsigned long long* __restrict__ hist, int pass,
                                     double* __restrict__ thr_out) {
    __shared__ unsigned long long h[256];
    h[threadIdx.x] = hist[threadIdx.x];
    hist[threadIdx.x] = 0ull;                                  // ready for the next pass
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long r = state[1];
        int bin = 0;
        for (; bin < 255; ++bin) {
            if (r < h[bin]) break;
            r -= h[bin];
        }
        state[1] = r;
        state[0] |= static_cast<unsigned long long>(bin) << (56 - 8 * pass);
        if (pass == 7) *thr_out = f64_unkey(state[0]);
    }
}
__global__ void anomaly_flags_kernel(const double* __restrict__ l2, long long n_show, const double* __restrict__ thr, uint8_t* __restrict__ flags) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n_show) flags[i] = ((1.0 - l2[i]) <= *thr) ? 1 : 0;
}

// ------------------------------------------------------------------ measurement helpers (bench.py)
// counter-based N(0,1): splitmix64 of (seed, global element index) -> two uniforms -> Box-Muller
__global__ void synthetic_normal_kernel(float* __restrict__ out, long long n, unsigned long long seed, unsigned long long elem0) {
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        unsigned long long z = seed * 0x9E3779B97F4A7C15ull + (elem0 + static_cast<unsigned long long>(i)) * 0xD1B54A32D192ED03ull + 0x632BE59BD9B4E019ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        const float u1 = (static_cast<float>(static_cast<unsigned>(z >> 40)) + 1.0f) * (1.0f / 16777217.0f);   // (0, 1)
        const float u2 = static_cast<float>(static_cast<unsigned>(z) >> 8) * (1.0f / 16777216.0f);
        out[i] = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
    }
}
// fp32 FMA roof: 16 independent fmaf chains per thread
__global__ void __launch_bounds__(256) fma_peak_kernel(float* __restrict__ sink, int iters, float seed) {
    float a[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) a[j] = seed + 0.001f * j + 1e-6f * threadIdx.x;
    const float m = 0.9999f, c = 1e-4f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int j = 0; j < 16; ++j) a[j] = __fmaf_rn(a[j], m, c);
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += a[j];
    if (s == 123.456f) *sink = s;      // never true: keeps the chains alive
}

// the same with packed fma.rn.f32x2 (FFMA2: two IEEE fp32 FMAs per instruction)
__global__ void __launch_bounds__(256) fma2_peak_kernel(float* __restrict__ sink, int iters, float seed) {
    unsigned long long a[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float2 v = make_float2(seed + 0.001f * j + 1e-6f * threadIdx.x, seed + 0.002f * j);
        a[j] = *reinterpret_cast<unsigned long long*>(&v);
    }
    float2 mv = make_float2(0.9999f, 0.9999f), cv = make_float2(1e-4f, 1e-4f);
    const unsigned long long m = *reinterpret_cast<unsigned long long*>(&mv), c = *reinterpret_cast<unsigned long long*>(&cv);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int j = 0; j < 8; ++j) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(a[j]) : "l"(m), "l"(c));
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { float2 v = *reinterpret_cast<float2*>(&a[j]); s += v.x + v.y; }
    if (s == 123.456f) *sink = s;
}

}  // namespace ganrev

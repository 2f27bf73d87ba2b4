// refine.cuh -- the CUDA-core pieces of noise-vector refinement (ganrev_refine_l2; DESIGN.md section 4.5):
//   * G's last conv (128 -> C, 3x3) + sigmoid + squared-L2 loss, backwards: e2 = [h2 > 0] * conv3^T(2 (y - x) y (1 - y))
//     (K = 9*C is far too thin for the MMA; the kernel is bound by the 256 B of h2 read and the 256 B of e2 written per pixel)
//   * Adam on z with the Gaussian prior and the optional clamp, optim.adam's update as ganrev_train_R_step applies it
// The convs conv2^T / conv1^T and Linear^T run on the tensor cores (conv_tc.cuh, MASKSUM epilogue / fp32-output Linear).
#pragma once
#include "common.cuh"

namespace ganrev {

// One thread per (pixel, 8 consecutive channels): the 16 threads of a pixel read / write its 256 contiguous bytes of h2 / e2.
// w3t: fp32 [tap = ky*3 + kx][COUT][128] forward weights.  e3 of the output pixel (oy, ox) = (iy + 1 - ky, ix + 1 - kx) is
// recomputed from y and x by every thread that needs it (cached loads); taps are added in (ky, kx, co) order -- a fixed order.
template <int COUT>
__global__ void __launch_bounds__(256)
g_conv3_adjoint_kernel(const float* __restrict__ y, const float* __restrict__ x, const float* __restrict__ w3t,
                       const bf16* __restrict__ h2, bf16* __restrict__ e2, int H, int W, int lgH, int lgW, long long n_img) {
    __shared__ __align__(16) float ws[9 * COUT * 128];
    for (int i = threadIdx.x; i < 9 * COUT * 128; i += blockDim.x) ws[i] = w3t[i];
    __syncthreads();
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long pix = t >> 4;
    const int c0 = static_cast<int>(t & 15) * 8;
    if (pix >= (n_img << (lgH + lgW))) return;
    const int ix = static_cast<int>(pix) & (W - 1);
    const int iy = static_cast<int>(pix >> lgW) & (H - 1);
    const long long n = pix >> (lgH + lgW);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.0f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int oy = iy + 1 - ky;
        if (oy < 0 || oy >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int ox = ix + 1 - kx;
            if (ox < 0 || ox >= W) continue;
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                const long long off = ((n * COUT + co) << (lgH + lgW)) + (static_cast<long long>(oy) << lgW) + ox;
                const float yv = __ldg(y + off), xv = __ldg(x + off);
                const float e = __fmul_rn(__fmul_rn(2.0f * (yv - xv), yv), 1.0f - yv);   // d/d(pre-sigmoid) of (y - x)^2
                const float4* wr = reinterpret_cast<const float4*>(ws + ((ky * 3 + kx) * COUT + co) * 128 + c0);
                const float4 wa = wr[0], wb = wr[1];
                acc[0] += wa.x * e; acc[1] += wa.y * e; acc[2] += wa.z * e; acc[3] += wa.w * e;
                acc[4] += wb.x * e; acc[5] += wb.y * e; acc[6] += wb.z * e; acc[7] += wb.w * e;
            }
        }
    }
    const uint4 hv = __ldg(reinterpret_cast<const uint4*>(h2 + pix * 128 + c0));
    const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {   // ReLU mask: bf16 > 0 (sign bit clear, not +0)
        const uint32_t lo = hw[k] & 0xFFFFu, hi = hw[k] >> 16;
        const float a = (lo != 0u && lo < 0x8000u) ? acc[2 * k] : 0.0f, b = (hi != 0u && hi < 0x8000u) ? acc[2 * k + 1] : 0.0f;
        __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
        o[k] = *reinterpret_cast<uint32_t*>(&v);
    }
    __stcg(reinterpret_cast<uint4*>(e2 + pix * 128 + c0), make_uint4(o[0], o[1], o[2], o[3]));
}

struct RefineHyper { float beta1, beta2, eps, prior2, zclamp, step_size; };   // prior2 = 2 * prior; step_size per iteration (host)

// grad = W_lin^T (s0 e0) + 2 prior z  (ganrev_debug_refine_grad; the same float operations as refine_adam_kernel)
__global__ void refine_grad_kernel(const float* __restrict__ glin, const float* __restrict__ z, float prior2, float* __restrict__ grad, long long n) {
    const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e < n) grad[e] = __fadd_rn(glin[e], __fmul_rn(prior2, z[e]));
}

// One Adam step on z in place (train.cuh adam_kernel's update, with the prior term instead of the L1 / L2 penalties), then the clamp.
__global__ void refine_adam_kernel(float* __restrict__ z, const float* __restrict__ glin, float* __restrict__ m, float* __restrict__ v, long long n, RefineHyper h) {
    const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const float x = z[e];
    const float g = __fadd_rn(glin[e], __fmul_rn(h.prior2, x));
    const float mm = __fadd_rn(__fmul_rn(h.beta1, m[e]), __fmul_rn(1.0f - h.beta1, g));
    const float vv = __fadd_rn(__fmul_rn(h.beta2, v[e]), __fmul_rn(__fmul_rn(1.0f - h.beta2, g), g));
    m[e] = mm; v[e] = vv;
    float xn = __fsub_rn(x, __fdiv_rn(__fmul_rn(h.step_size, mm), __fadd_rn(__fsqrt_rn(vv), h.eps)));
    if (h.zclamp > 0.0f) xn = fminf(fmaxf(xn, -h.zclamp), h.zclamp);
    z[e] = xn;
}

}  // namespace ganrev

// common.cuh -- shared declarations for libganrev_cuda.so (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/ganrev.h"

namespace ganrev {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------
// Per-kernel profiling record (ganrev_profile_*): CUDA events on the library stream.
// ---------------------------------------------------------------------------------
struct ProfEntry {
    std::string name;
    uint64_t launches = 0;
    double total_ms = 0.0;
    double flops = 0.0;   // algorithmic-executed FLOPs summed over launches
    double bytes = 0.0;   // algorithmic bytes summed over launches
};
struct ProfPending {
    int entry;
    cudaEvent_t e0, e1;
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;  // bytes
};

// conv-as-GEMM layer description, shared by the tcgen05 kernel and the CUDA-core kernel.
//
// K loop: per item, `units` = ngroups * cin_chunks units; unit (g, cc) covers tap group g (one
// horizontal offset gdx with ndy consecutive vertical offsets gdy0 .. gdy0+ndy-1) and input
// channels [64*cc, 64*cc+64).  Weight K index = ((g*ndy + j)*Cin + ci).  With ndy > 1 the A
// operand of a unit is ONE box of BH+ndy-1 rows; the ndy vertical taps are 1024B-aligned
// offsets into it (halo reuse).  ndy == 1 expresses arbitrary tap lists (one tap per group).
struct ConvGemm {
    // A operand: NHWC bf16 activation [n_cap][Hin][Win][Cin]; M tile = box (64ch, BW, BH(+ndy-1), BN)
    int Hin, Win, Cin;
    int lgBW, lgBH, lgBN;      // log2 of the M-tile extents, BW*BH*BN == 128
    int tiles_w, tiles_h;      // tiles per image (powers of two: H, W are)
    int lgTW, lgTH;            // log2 of the above
    int lgNT;                  // log2(n_tiles), or -1 when n_tiles is not a power of two
    int total_tiles;           // M tiles in this launch
    int n_img;                 // valid images in this launch
    int nphase, ngroups, ndy;  // phase-decomposed upsample: 4 phases; else 1
    int8_t gdx[4][9], gdy0[4][9];
    int cin_chunks, units, ups, stages;
    int a_unit_bytes, b_kb_bytes, unit_bytes, stage_bytes, dy_stride_bytes;
    // B operand: bf16 weights [nphase*cout_pad][ngroups*ndy*Cin]
    int cout_pad, n_tiles;     // cout_pad = n_tiles*NT
    int cout_real;             // channels actually stored
    long long out_sN;          // output strides (elements): image,
    int out_sP, out_sC;        //   pixel (row-major oh*Wout+ow), channel.  bf16 NHWC: (H*W*C, C, 1); fp32 NCHW: (C*H*W, 1, H*W)
    int Hout, Wout, up, pool, act, out_fp32;
    int tma_hybrid;            // TMA-store epilogue: first chunk of each round by st.global, second by TMA (no wait on the staging buffer)
    int xpose2;                // two store-transpose buffers per epilogue warp (TMA-store epilogue: one store may still be reading)
    int tma_store;             // bf16 NHWC output written by TMA bulk tensor stores (plain convs / linears); else st.global
    float post_scale;
    void* out;
    const float* shift;        // [cout_pad] folded BN shift (+ conv bias); the BN scale is folded into B
    const bf16* A;             // raw pointers (CUDA-core kernel)
    const bf16* B;
    int* err_flag;
    long long* trace;          // optional clock64 timeline of CTA 0 (ganrev_debug_trace), [8 roles][256 events]
    int dbg;                   // timing experiments only: bit0 skip A loads, bit1 skip B loads, bit2 skip epilogue, bit3 skip MMAs
    // FUSE3 variants (G's Up+Conv 256->128 with the tap products of the last conv, models.lua:132, computed in the epilogue):
    const float* w3;           // fp32 [9*C][128] (tap, output channel)-major weights of the 128 -> C conv; the activation itself is never stored
    int w3_c;                  // C (1 or 3)
    float* taps;               // fp32 planes P[tap*C + co][pixel] (pixel = (n*Hout + oh)*Wout + ow), read by g_conv3_gather_kernel
    long long taps_plane;      // floats per plane
    // MASKSUM variants (G's backward convs, refinement): bf16 tensor with exactly the output's layout; output = 2x2 sum-pool * [ref > 0]
    const bf16* ref;
};

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_ELU = 2, ACT_TANH = 3, ACT_SIGMOID = 4 };

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == ACT_RELU) return v > 0.0f ? v : 0.0f;
    if (act == ACT_ELU) return v > 0.0f ? v : expm1f(v);
    if (act == ACT_TANH) return tanhf(v);
    if (act == ACT_SIGMOID) return 1.0f / (1.0f + expf(-v));
    return v;
}

// nn.ELU(alpha=1) for bf16 outputs: exp via one ex2.approx (abs error ~2e-7, below the bf16
// rounding of anything that matters next to O(1e-3)+ activations); 4 instructions per element.
__device__ __forceinline__ float elu_fast(float v) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v * 1.4426950408889634f));
    e -= 1.0f;
    return v > 0.0f ? v : e;
}

}  // namespace ganrev

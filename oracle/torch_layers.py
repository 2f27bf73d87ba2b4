"""fp64 references of G's and R's forward layers one at a time (ganrev_debug_G_stage / ganrev_debug_R_stage), in PyTorch-CPU.

Each reference takes the library's own input to the layer (its bf16 activation, as fp64 values) and weights rounded exactly as
the library rounds them, and returns (ref, tot): the fp64 result and the fp64 sum of absolute terms (products, plus the folded
bias), which bounds what a different fp32 / tensor-core accumulation order can change.  ReLU / ELU layers take `act=False` to
return the pre-activation (after the max-pool where there is one: max commutes with both).  Tests and tools only; never the
product.

The library's roundings, restated (csrc/ganrev.cu, conv1_tc.cuh):
  * fold_bn, in float32: s = g / sqrt(v + 1e-5), shift = beta + (bias - mean) * s.
  * Linear weights (build_tc_layer, KIND_LINEAR): f2bf(float32(w * s)), both operands float32.  G's Linear rows are permuted from
    View(512, H/4, W/4) to NHWC (fn = s*512 + c <- fo = c*HW0 + s); R Linear1's columns the same way (s*128 + c <- c*HWq + s),
    with SpatialDropout's x0.75 multiplied in first, in float32: f2bf(float32(float32(0.75 * w) * s)).  R Linear2 and G's tap
    GEMM have s = 1: f2bf(w).
  * Conv and phase weights (KIND_CONV3 / KIND_UPCONV3): f2bf(float32(double_sum * double(s))).  A 3x3 conv's sum is the one tap;
    a phase tap of upsample+conv sums w over build_tc_layer's S[a][t] rows x S[b][t] columns, in ky-then-kx order, in double.
  * G's Linear input is __float2bfloat16_rn(noise) (zero-padded to kpad: the padding adds nothing).
  * R conv1 on the tensor cores (conv1_tc.cuh): weights f2bf(float32(w * s)), used twice; every tap x (0 where the dropout mask
    byte is 0, or outside the image) is split into hi = x with its low 16 bits cleared (a bf16 value, exactly) and
    lo = x - hi (exact in float32) with its low 16 bits cleared too (truncated, not rounded), so the product is (hi + lo) * w.
    The CUDA-core conv1 (conv_impl 1) keeps float32 x and w and applies ELU(acc * s + shift).
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle.torch_grad import EPS, bf16_to_f32, f2bf

f32, f64 = np.float32, np.float64
# build_tc_layer's S[a][t] = {first, last} kernel row (column) of phase a's tap t
S = (((0, 0), (1, 2)), ((0, 1), (2, 2)))


def bf(a):
    """float32 values through the library's host f2bf, as fp64."""
    return bf16_to_f32(f2bf(np.asarray(a, f32))).astype(f64)


def bits(b):
    """Stored bf16 activations (uint16 bits) as fp64 values."""
    return bf16_to_f32(b).astype(f64)


def relu(v):
    return np.maximum(v, 0.0)


def elu(v):
    return np.where(v > 0, v, np.expm1(np.minimum(v, 0.0)))


def fold_bn(p, bias, bn, rounded=True):
    """(scale, shift): float32 as fold_bn computes them (returned as fp64), or exact in fp64."""
    if rounded:
        s = p[bn + ".g"].astype(f32) / np.sqrt(p[bn + ".v"].astype(f32) + f32(EPS))
        return s.astype(f64), (p[bn + ".b"] + (bias.astype(f32) - p[bn + ".m"]) * s).astype(f64)
    s = p[bn + ".g"].astype(f64) / np.sqrt(p[bn + ".v"].astype(f64) + EPS)
    return s, p[bn + ".b"].astype(f64) + (bias.astype(f64) - p[bn + ".m"].astype(f64)) * s


def _round_prod(w64, s64, rounded):
    """f2bf(float32(double w * double s)) (rounded) or the fp64 product."""
    prod = w64 * s64
    return bf(prod.astype(f32)) if rounded else prod


# ---------------------------------------------------------------- weights, as the library holds them
def g_weights(p, C, H, W, nd, rounded=True):
    """{layer: (weights, shift)}: lin [F][nd] (NHWC rows), c1 / c2 phase filters [2][2][co][ci][2][2] (phase a, b; tap ty, tx),
    taps [9C][128] (row t*C + co: bf16, the unfused 1x1 GEMM), w3 [9C][128] float32 (the fused epilogue), b3 [C]."""
    hw0 = (H // 4) * (W // 4)
    perm = lambda a: a.reshape((512, hw0) + a.shape[1:]).swapaxes(0, 1).reshape((512 * hw0,) + a.shape[1:])
    s0, sh0 = fold_bn(p, p["lin.b"], "bn0", rounded)
    lw = perm(p["lin.w"])
    s0, sh0 = perm(s0), perm(sh0)
    if rounded:
        lin = bf(lw.astype(f32) * s0.astype(f32)[:, None])
    else:
        lin = lw.astype(f64) * s0[:, None]
    out = {"lin": (lin, sh0)}
    for layer, bn in (("c1", "bn1"), ("c2", "bn2")):
        s, sh = fold_bn(p, p[layer + ".b"], bn, rounded)
        out[layer] = (phase_weights(p[layer + ".w"], s, rounded), sh)
    w3 = p["c3.w"]                                                     # [C][128][3][3]
    t = w3.reshape(C, 128, 9).transpose(2, 0, 1).reshape(9 * C, 128)     # row t*C + co
    out["taps"] = (bf(t) if rounded else t.astype(f64), np.zeros(9 * C))
    out["w3"] = t.astype(f64)
    out["b3"] = p["c3.b"].astype(f64)
    return out


def phase_weights(w, s, rounded=True):
    """Upsample x2 + 3x3 conv as four 2x2 convs on the low-resolution input: [a][b][co][ci][ty][tx] =
    f2bf(float32(sum over S[a][ty] x S[b][tx] of w, in double, * s[co]))."""
    w = np.asarray(w, f64)
    co, ci = w.shape[:2]
    out = np.empty((2, 2, co, ci, 2, 2))
    for a in range(2):
        for b in range(2):
            for ty in range(2):
                for tx in range(2):
                    acc = np.zeros((co, ci))
                    for ky in range(S[a][ty][0], S[a][ty][1] + 1):
                        for kx in range(S[b][tx][0], S[b][tx][1] + 1):
                            acc = acc + w[:, :, ky, kx]
                    out[a, b, :, :, ty, tx] = _round_prod(acc, np.asarray(s, f64)[:, None], rounded)
    return out


def r_weights(p, C, H, W, nd, rounded=True):
    """{layer: (weights, shift)}: c1..c6 [co][ci][3][3] (c1: the tensor-core weights), l1 [512][F] (NHWC columns, x0.75 folded),
    out [nd][512]; and c1_simt = (float32 w, scale, shift) of the CUDA-core conv1."""
    out = {}
    for i in range(1, 7):
        s, sh = fold_bn(p, p[f"c{i}.b"], f"bn{i}", rounded)
        w = p[f"c{i}.w"]
        if i == 1 and rounded:   # conv1 pack: f2bf(w * s), both float32
            wr = bf(w.astype(f32) * s.astype(f32)[:, None, None, None])
        else:
            wr = _round_prod(w.astype(f64), s[:, None, None, None], rounded)
        out[f"c{i}"] = (wr, sh)
        if i == 1:
            out["c1_simt"] = (w.astype(f64), s, sh)
    hwq = (H // 4) * (W // 4)
    l1 = p["l1.w"].reshape(512, 128, hwq).swapaxes(1, 2).reshape(512, 128 * hwq)   # column s*128 + c <- c*hwq + s
    s7, sh7 = fold_bn(p, p["l1.b"], "bn7", rounded)
    if rounded:
        out["l1"] = (bf((f32(0.75) * l1.astype(f32)) * s7.astype(f32)[:, None]), sh7)
    else:
        out["l1"] = (0.75 * l1.astype(f64) * s7[:, None], sh7)
    out["out"] = (bf(p["l2.w"]) if rounded else p["l2.w"].astype(f64), p["l2.b"].astype(f64))
    return out


# ---------------------------------------------------------------- layers
def _nchw(a):
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, f64).transpose(0, 3, 1, 2)))


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous().numpy()


def ref_linear(x, w, shift):
    """x [N][K] times w [O][K] plus shift: (value, sum of |products| + |shift|)."""
    x = np.asarray(x, f64).reshape(len(x), -1)
    return x @ w.T + shift, np.abs(x) @ np.abs(w).T + np.abs(shift)


def ref_g_lin(noise, w, shift, H, W, act=True, rounded=True):
    """G Linear + BN + ReLU on __float2bfloat16_rn(noise): [N][H/4][W/4][512]."""
    x = bf(noise) if rounded else np.asarray(noise, f64)
    v, t = ref_linear(x, w, shift)
    shape = (len(x), H // 4, W // 4, 512)
    return (relu(v) if act else v).reshape(shape), t.reshape(shape)


def ref_upconv(h, wph, shift, act=True):
    """Upsample x2 + conv 3x3 + BN + ReLU in phase form on h [N][h][w][ci]: output pixel (2y + a, 2x + b) is the 2x2 conv of phase
    (a, b) over low-resolution rows y + a - 1 + ty, columns x + b - 1 + tx (zero outside).  Returns NHWC [N][2h][2w][co]."""
    hp = F.pad(_nchw(h), (1, 1, 1, 1))
    N, _, hh, ww = hp.shape
    hh, ww = hh - 2, ww - 2
    co = wph.shape[2]
    val, tot = torch.empty(N, co, 2 * hh, 2 * ww, dtype=torch.float64), torch.empty(N, co, 2 * hh, 2 * ww, dtype=torch.float64)
    for a in range(2):
        for b in range(2):
            src = hp[:, :, a:a + hh + 1, b:b + ww + 1]
            wt = torch.from_numpy(np.ascontiguousarray(wph[a, b]))
            val[:, :, a::2, b::2] = F.conv2d(src, wt)
            tot[:, :, a::2, b::2] = F.conv2d(src.abs(), wt.abs())
    sh = torch.from_numpy(np.asarray(shift, f64))[None, :, None, None]
    v, t = _nhwc(val + sh), _nhwc(tot + sh.abs())
    return (relu(v) if act else v), t


def ref_conv3(h, w, shift, pool=False, act=True, nchw_in=False):
    """3x3 / pad 1 conv + BN (+ 2x2 max-pool) + ELU on h [N][H][W][ci] (nchw_in: [N][ci][H][W]).  Pooled: the max of the four
    pre-activations, with the largest sum of |terms| of the window.  Returns NHWC."""
    x = torch.from_numpy(np.ascontiguousarray(h, f64)) if nchw_in else _nchw(h)
    wt = torch.from_numpy(np.ascontiguousarray(w, f64))
    sh = torch.from_numpy(np.asarray(shift, f64))[None, :, None, None]
    val = F.conv2d(x, wt, padding=1) + sh
    tot = F.conv2d(x.abs(), wt.abs(), padding=1) + sh.abs()
    if pool:
        val, tot = F.max_pool2d(val, 2), F.max_pool2d(tot, 2)
    v, t = _nhwc(val), _nhwc(tot)
    return (elu(v) if act else v), t


def conv1_input(x, mask=None, split=True):
    """R conv1's operand for images x [N][C][H][W] float32: x where the mask byte is non-zero (else 0); split: hi + lo as
    conv1_tc.cuh forms them (hi = x & 0xFFFF0000, lo = (x - hi) & 0xFFFF0000, bit patterns), as fp64."""
    x = np.ascontiguousarray(x, f32)
    if mask is not None:
        x = np.where(np.asarray(mask) != 0, x, f32(0.0))
    if not split:
        return x.astype(f64)
    hi = (x.view(np.uint32) & np.uint32(0xFFFF0000)).view(f32)
    lo = np.ascontiguousarray(x - hi)
    lo = (lo.view(np.uint32) & np.uint32(0xFFFF0000)).view(f32)
    return hi.astype(f64) + lo.astype(f64)


def ref_r_conv1(x_eff, w, shift, act=True):
    """R conv1 + BN + ELU (tensor cores) on conv1_input's operand [N][C][H][W]: NHWC [N][H][W][64]."""
    return ref_conv3(x_eff, w, shift, act=act, nchw_in=True)


def ref_r_conv1_simt(x, w, s, shift, act=True):
    """The CUDA-core conv1 (conv_impl 1): ELU(conv(x, w) * s + shift), x float32 (masked, not split), w float32."""
    xt = torch.from_numpy(np.ascontiguousarray(x, f64))
    wt = torch.from_numpy(np.ascontiguousarray(w, f64))
    s_, sh = (torch.from_numpy(np.asarray(a, f64))[None, :, None, None] for a in (s, shift))
    val = F.conv2d(xt, wt, padding=1) * s_ + sh
    tot = F.conv2d(xt.abs(), wt.abs(), padding=1) * s_.abs() + sh.abs()
    v, t = _nhwc(val), _nhwc(tot)
    return (elu(v) if act else v), t


def ref_taps_unfused(h2, wt):
    """The 1x1 tap GEMM on the stored h2 [N][H][W][128] with bf16 weights wt [9C][128]: fp32 planes [N][9C][H][W]."""
    N, H, W, _ = h2.shape
    v, t = ref_linear(np.asarray(h2, f64).reshape(N * H * W, 128), wt, 0.0)
    tr = lambda a: a.reshape(N, H, W, -1).transpose(0, 3, 1, 2)
    return tr(v), tr(t)


def ref_taps_fused(pre2, tot2, w3):
    """Tap products out of G conv2's epilogue: relu(conv2) -- not rounded to bf16 -- times the float32 w3 [9C][128].  pre2 / tot2:
    ref_upconv(..., act=False) of conv2 on the library's c1.  The sum of |terms| carries conv2's own: sum_ci |w3| tot2[ci], which
    bounds both conv2's accumulation error seen through w3 and the fp32 products here (|relu(pre2)| <= tot2)."""
    N, H, W, _ = pre2.shape
    r = relu(pre2).reshape(N * H * W, 128)
    v = r @ w3.T
    t = tot2.reshape(N * H * W, 128) @ np.abs(w3).T
    tr = lambda a: a.reshape(N, H, W, -1).transpose(0, 3, 1, 2)
    return tr(v), tr(t)


def ref_y(taps, b3, C):
    """g_conv3_gather_kernel on the library's taps [N][9C][H][W]: y[co] = sigmoid(b3[co] + sum over (ky, kx) of plane
    (ky*3 + kx)*C + co at pixel (y + ky - 1, x + kx - 1), zero outside).  Returns (y [N][C][H][W], |b3| + sum |taps|)."""
    P = np.asarray(taps, f64)
    N, _, H, W = P.shape
    acc = np.zeros((N, C, H, W)) + b3[None, :, None, None]
    tot = np.zeros((N, C, H, W)) + np.abs(b3)[None, :, None, None]
    for ky in range(3):
        for kx in range(3):
            pl = P[:, (ky * 3 + kx) * C:(ky * 3 + kx + 1) * C]
            sh = np.zeros_like(pl)
            y0, y1, x0, x1 = max(0, 1 - ky), min(H, H + 1 - ky), max(0, 1 - kx), min(W, W + 1 - kx)
            sh[:, :, y0:y1, x0:x1] = pl[:, :, y0 + ky - 1:y1 + ky - 1, x0 + kx - 1:x1 + kx - 1]
            acc += sh
            tot += np.abs(sh)
    return 1.0 / (1.0 + np.exp(-acc)), tot


def ref_r_l1(c6, w, shift, act=True):
    """R Linear1 + BN + ELU on the pooled conv6 [N][H/4][W/4][128] (flattened NHWC): [N][512]."""
    v, t = ref_linear(np.asarray(c6, f64).reshape(len(c6), -1), w, shift)
    return (elu(v) if act else v), t


def ref_r_out(l1, w, b, tanh=False):
    """R Linear2 (+ Tanh), fp32 out: [N][nd]."""
    v, t = ref_linear(l1, w, b)
    return (np.tanh(v) if tanh else v), t

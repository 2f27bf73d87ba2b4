"""Gradient of the refinement objective f(z) = ||G(z) - x||^2 + prior ||z||^2 (ganrev_refine_l2), two ways, in PyTorch-CPU:

  * autograd through G3 (models.lua:104-143) written with torch.nn.functional, grad-enabled;
  * the closed form the CUDA kernels implement (DESIGN.md section 4.5): BN folded (s = per-channel scale),
      e3 = 2 (y - x) y (1 - y),  e2 = [h2 > 0] conv3^T(e3),  e1 = [h1 > 0] sumpool2x2(conv2^T(e2)),
      e0 = [h0 > 0] sumpool2x2(conv1^T(e1)),  grad = W_lin^T (s0 e0) + 2 prior z,
    with conv^T a plain 3x3 convolution at the high resolution (weights W^T[ci][2-ky][2-kx][co] s[co]) and the Linear's
    transpose taken in the NHWC feature order the library's forward Linear emits.

`p` is the parameter dict of weights.unpack(blob, weights.g_layout(...)).  Tests and tools only; never the product.

Per-stage references (`ref_e2`, `ref_masksum`, `ref_glin`): each backward kernel of the library on its own.  They take the library's
own input to that stage (its bf16 activations and gradients), weights rounded exactly as the library rounds them
(`conv_t_weights`, `linear_t_weights`), and return the fp64 result together with the fp64 sum of absolute products, which bounds
what a different accumulation order can change.  With `rounded=False` / `exact=True` and fp64 inputs they compose to
`adjoint_grad` (tests/test_refine_cpu.py), which pins their conventions (flip, transpose, NHWC order, permutation) on the CPU.
"""
import numpy as np
import torch
import torch.nn.functional as F

EPS = 1e-5


def _t(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype)


def _bn(x, p, name, dtype):
    return F.batch_norm(x, _t(p[name + ".m"], dtype), _t(p[name + ".v"], dtype), _t(p[name + ".g"], dtype),
                        _t(p[name + ".b"], dtype), training=False, eps=EPS)


def forward_G(p, C, H, W, nd, z, dtype=torch.float32):
    """G3 in eval mode, differentiable in z (a torch tensor).  Returns (y, h0, h1, h2) with h the post-ReLU activations (NCHW)."""
    x = F.linear(z, _t(p["lin.w"], dtype), _t(p["lin.b"], dtype))
    h0 = F.relu(_bn(x, p, "bn0", dtype)).view(-1, 512, H // 4, W // 4)
    x = F.interpolate(h0, scale_factor=2, mode="nearest")
    h1 = F.relu(_bn(F.conv2d(x, _t(p["c1.w"], dtype), _t(p["c1.b"], dtype), padding=1), p, "bn1", dtype))
    x = F.interpolate(h1, scale_factor=2, mode="nearest")
    h2 = F.relu(_bn(F.conv2d(x, _t(p["c2.w"], dtype), _t(p["c2.b"], dtype), padding=1), p, "bn2", dtype))
    y = torch.sigmoid(F.conv2d(h2, _t(p["c3.w"], dtype), _t(p["c3.b"], dtype), padding=1))
    return y, h0, h1, h2


def objective(p, C, H, W, nd, z, x, prior, dtype=torch.float32):
    """Per-image f(z) = ||G(z) - x||^2 + prior ||z||^2 (torch tensor [N])."""
    y = forward_G(p, C, H, W, nd, z, dtype)[0]
    return ((y - x) ** 2).flatten(1).sum(1) + prior * (z ** 2).sum(1)


def autograd_grad(p, C, H, W, nd, z, x, prior, dtype=torch.float32):
    """(grad [N x nd], f [N]) by autograd; every image's f depends on its own z only, so d(sum f)/dz is per-image grad."""
    zt = _t(z, dtype).requires_grad_(True)
    f = objective(p, C, H, W, nd, zt, _t(x, dtype), prior, dtype)
    f.sum().backward()
    return zt.grad.numpy(), f.detach().numpy()


def _scale(p, name):
    return p[name + ".g"].astype(np.float64) / np.sqrt(p[name + ".v"].astype(np.float64) + EPS)


def _conv_t(e, w, s, dtype):
    """conv^T of a forward 3x3 conv with weights w [co][ci][3][3] and BN scale s [co]: a plain 3x3 conv co -> ci."""
    wt = _t((w.astype(np.float64) * s[:, None, None, None]).transpose(1, 0, 2, 3)[:, :, ::-1, ::-1].copy(), dtype)
    return F.conv2d(e, wt, padding=1)


def adjoint_grad(p, C, H, W, nd, z, x, prior, dtype=torch.float64):
    """The closed form above (grad [N x nd])."""
    with torch.no_grad():
        zt, xt = _t(z, dtype), _t(x, dtype)
        y, h0, h1, h2 = forward_G(p, C, H, W, nd, zt, dtype)
        e3 = 2.0 * (y - xt) * y * (1.0 - y)
        w3 = _t(p["c3.w"].transpose(1, 0, 2, 3)[:, :, ::-1, ::-1].copy(), dtype)
        e2 = (h2 > 0).to(dtype) * F.conv2d(e3, w3, padding=1)
        e1 = (h1 > 0).to(dtype) * 4.0 * F.avg_pool2d(_conv_t(e2, p["c2.w"], _scale(p, "bn2"), dtype), 2)
        e0 = (h0 > 0).to(dtype) * 4.0 * F.avg_pool2d(_conv_t(e1, p["c1.w"], _scale(p, "bn1"), dtype), 2)
        hw0 = (H // 4) * (W // 4)
        e0n = e0.permute(0, 2, 3, 1).reshape(e0.shape[0], -1)                        # NHWC feature order: fn = s*512 + c
        perm = lambda a: a.reshape((512, hw0) + a.shape[1:]).swapaxes(0, 1).reshape((512 * hw0,) + a.shape[1:])   # from fo = c*hw0 + s
        s0 = _t(perm(_scale(p, "bn0")), dtype)
        wl = _t(perm(p["lin.w"].astype(np.float64)), dtype)                         # [F (NHWC)][nd]
        return ((e0n * s0) @ wl + 2.0 * prior * zt).numpy()


# ---------------------------------------------------------------- per-stage references (bf16 conventions of the library)
def f2bf(a):
    """bf16 bits (uint16) of float32 values, round-to-nearest-even, NaN preserved (quiet): the library's host f2bf."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    return np.where(nan, ((u >> 16) | 0x40).astype(np.uint16), r)


def bf16_to_f32(bits):
    return (np.asarray(bits, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


def bf16_rne(a):
    """float64 values rounded once to the nearest bf16 (ties to even), as float64.  No detour through float32 (that would round
    twice); the normal bf16 range is assumed (|a| >= 2^-126 or 0), which every stage value that survives its mask is in."""
    u = np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)
    low = np.uint64((1 << 45) - 1)                     # float64 keeps 52 fraction bits, bf16 keeps 7
    r = (u + np.uint64((1 << 44) - 1) + ((u >> np.uint64(45)) & np.uint64(1))) & ~low
    return r.view(np.float64)


def ulp_bf16(a):
    """Spacing of bf16 numbers at |a| (the smallest normal spacing at 0)."""
    e = np.floor(np.log2(np.maximum(np.abs(np.asarray(a, np.float64)), 2.0 ** -126)))
    return np.exp2(e - 7)


def bf16_mask(bits):
    """[h > 0] of stored bf16 activations: sign bit clear and not +0."""
    b = np.asarray(bits, dtype=np.uint16)
    return (b != 0) & (b < 0x8000)


def _scale32(p, name):
    """fold_bn's float32 scale g / sqrtf(v + 1e-5f)."""
    g, v = p[name + ".g"].astype(np.float32), p[name + ".v"].astype(np.float32)
    return g / np.sqrt(v + np.float32(EPS))


def conv_t_weights(p, layer, rounded=True):
    """Weights [ci][co][3][3] (fp64) of the plain 3x3 conv co -> ci that is conv^T of G's `layer` ("c1" / "c2") with its BN scale
    folded: flipped and transposed.  rounded: bf16(float32(w * float32 s)), as the library's backward layers hold them;
    otherwise w * s in fp64."""
    bn = {"c1": "bn1", "c2": "bn2"}[layer]
    w = p[layer + ".w"]
    if rounded:
        ws = bf16_to_f32(f2bf(w * _scale32(p, bn)[:, None, None, None])).astype(np.float64)
    else:
        ws = w.astype(np.float64) * _scale(p, bn)[:, None, None, None]
    return ws.transpose(1, 0, 2, 3)[:, :, ::-1, ::-1].copy()


def linear_t_weights(p, H, W, nd, rounded=True):
    """[F][nd] (fp64): row fn = s*512 + c (the NHWC feature order of G's Linear output) holds W_lin[fo][:] * s0[fo], fo = c*HW0 + s
    (View(512, H/4, W/4)).  rounded: bf16(float32(w * float32 s0)), as the library's Linear^T holds it."""
    hw0 = (H // 4) * (W // 4)
    if rounded:
        wl = bf16_to_f32(f2bf(p["lin.w"] * _scale32(p, "bn0")[:, None])).astype(np.float64)
    else:
        wl = p["lin.w"].astype(np.float64) * _scale(p, "bn0")[:, None]
    return wl.reshape(512, hw0, nd).swapaxes(0, 1).reshape(512 * hw0, nd).copy()


def _nchw(a):
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, np.float64).transpose(0, 3, 1, 2)))


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous().numpy()


def ref_e2(y, x, w3, mask2, exact=False):
    """g_conv3_adjoint_kernel: e2 = [h2 > 0] conv3^T(e3), NHWC [N][H][W][128].  y, x: NCHW; w3: [C][128][3][3]; mask2: NHWC bool.
    e3 = ((2 (y - x)) y)(1 - y) with every operation rounded to float32 as the kernel computes it (exact: in fp64).
    Returns (e2 before bf16 rounding, sum of |products|), both fp64 and zero where the mask is off."""
    if exact:
        y64, x64 = np.asarray(y, np.float64), np.asarray(x, np.float64)
        e3 = 2.0 * (y64 - x64) * y64 * (1.0 - y64)
    else:
        y32, x32 = np.asarray(y, np.float32), np.asarray(x, np.float32)
        one = np.float32(1.0)
        e3 = ((np.float32(2.0) * (y32 - x32)) * y32) * (one - y32)
    e3 = torch.from_numpy(np.asarray(e3, np.float64))
    wt = w3.astype(np.float64).transpose(1, 0, 2, 3)[:, :, ::-1, ::-1].copy()
    val = F.conv2d(e3, torch.from_numpy(wt), padding=1)
    tot = F.conv2d(e3.abs(), torch.from_numpy(np.abs(wt)), padding=1)
    m = np.asarray(mask2, bool)
    return np.where(m, _nhwc(val), 0.0), np.where(m, _nhwc(tot), 0.0)


def ref_masksum(e, wt, mask):
    """The MASKSUM conv (conv2^T / conv1^T): [h > 0] sumpool2x2(conv3x3(e, wt)).  e: NHWC at the high resolution; wt: [ci][co][3][3]
    from conv_t_weights; mask: NHWC bool at half the resolution.  Returns (value, sum of |products|), fp64, zero where masked."""
    wt = torch.from_numpy(np.asarray(wt, np.float64))
    et = _nchw(e)
    val = 4.0 * F.avg_pool2d(F.conv2d(et, wt, padding=1), 2)
    tot = 4.0 * F.avg_pool2d(F.conv2d(et.abs(), wt.abs(), padding=1), 2)
    m = np.asarray(mask, bool)
    return np.where(m, _nhwc(val), 0.0), np.where(m, _nhwc(tot), 0.0)


def ref_glin(e0, wl):
    """Linear^T: e0 [N][F] (NHWC feature order) times wl [F][nd] (linear_t_weights).  Returns (value, sum of |products|), fp64."""
    e0 = np.asarray(e0, np.float64).reshape(len(e0), -1)
    return e0 @ wl, np.abs(e0) @ np.abs(wl)

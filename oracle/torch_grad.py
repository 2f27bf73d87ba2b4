"""Gradient of the refinement objective f(z) = ||G(z) - x||^2 + prior ||z||^2 (ganrev_refine_l2), two ways, in PyTorch-CPU:

  * autograd through G3 (models.lua:104-143) written with torch.nn.functional, grad-enabled;
  * the closed form the CUDA kernels implement (DESIGN.md section 4.5): BN folded (s = per-channel scale),
      e3 = 2 (y - x) y (1 - y),  e2 = [h2 > 0] conv3^T(e3),  e1 = [h1 > 0] sumpool2x2(conv2^T(e2)),
      e0 = [h0 > 0] sumpool2x2(conv1^T(e1)),  grad = W_lin^T (s0 e0) + 2 prior z,
    with conv^T a plain 3x3 convolution at the high resolution (weights W^T[ci][2-ky][2-kx][co] s[co]) and the Linear's
    transpose taken in the NHWC feature order the library's forward Linear emits.

`p` is the parameter dict of weights.unpack(blob, weights.g_layout(...)).  Tests and tools only; never the product.
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

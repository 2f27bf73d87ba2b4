"""References for face completion (ganrev_refine_masked_l2): the masked objective f(z) = sum over m = 1 of (G(z) - x)^2 + prior ||z||^2,
m a uint8 / bool keep-mask shaped like x (1 = keep).  Built on oracle/torch_grad.py, which states the unmasked objective; tests only.

  * `objective` / `autograd_grad`: autograd through G3 with the residual selected (torch.where), and x selected before the
    subtraction, so x under m = 0 (even NaN / Inf) reaches neither f nor its gradient.
  * `adjoint_grad` / `ref_e2`: the closed form and the per-stage reference of g_conv3_adjoint_kernel<C, true>, in which
    e3 = [m] 2 (y - x) y (1 - y).  Both call oracle/torch_grad.py's function with x replaced by y at m = 0: there
    e3 = 2 (y - y) y (1 - y) is exactly 0 (y is finite, in (0, 1)), in fp32 and in fp64, and so is its share of the sum of |products|.
    That is the masked e3 without restating the closed form.
"""
import numpy as np
import torch

from oracle import torch_grad as tg


def _keep(mask):
    return np.ascontiguousarray(mask) != 0


def objective(p, C, H, W, nd, z, x, prior, mask, dtype=torch.float32):
    """Per-image masked f(z) (torch tensor [N]); z and x are torch tensors."""
    y = tg.forward_G(p, C, H, W, nd, z, dtype)[0]
    keep = torch.from_numpy(_keep(mask))
    r = torch.where(keep, y - torch.where(keep, x, torch.zeros_like(x)), torch.zeros_like(y))
    return (r ** 2).flatten(1).sum(1) + prior * (z ** 2).sum(1)


def autograd_grad(p, C, H, W, nd, z, x, prior, mask, dtype=torch.float32):
    """(grad [N x nd], f [N]) of the masked objective by autograd."""
    zt = tg._t(z, dtype).requires_grad_(True)
    f = objective(p, C, H, W, nd, zt, tg._t(x, dtype), prior, mask, dtype)
    f.sum().backward()
    return zt.grad.numpy(), f.detach().numpy()


def adjoint_grad(p, C, H, W, nd, z, x, prior, mask, dtype=torch.float64):
    """The closed form with e3 = [m] e3 (grad [N x nd])."""
    with torch.no_grad():
        y = tg.forward_G(p, C, H, W, nd, tg._t(z, dtype), dtype)[0].numpy()
    return tg.adjoint_grad(p, C, H, W, nd, z, np.where(_keep(mask), np.asarray(x, y.dtype), y), prior, dtype)


def ref_e2(y, x, w3, mask2, mask, exact=False):
    """tg.ref_e2 for g_conv3_adjoint_kernel<C, true>: e3 is 0 where mask = 0, in the value and in the sum of |products|."""
    y = np.asarray(y, np.float32)
    return tg.ref_e2(y, np.where(_keep(mask), np.asarray(x, np.float32), y), w3, mask2, exact=exact)

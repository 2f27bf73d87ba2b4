"""The closed-form gradient the refinement kernels implement (flipped-weight 3x3 convs at the high resolution, 2x2 sum-pools,
ReLU masks, BN folded, the Linear transposed in NHWC feature order; oracle/torch_grad.py) equals autograd through G3."""
import numpy as np
import pytest

from oracle import torch_grad


@pytest.mark.parametrize("geom", [(1, 16, 16, 32), (1, 32, 32, 100), (3, 64, 64, 64)], ids=lambda g: "C%dx%dx%d_nd%d" % g)
@pytest.mark.parametrize("prior", [0.0, 0.05])
def test_adjoint_matches_autograd(pkg, geom, prior):
    import torch
    C, H, W, nd = geom
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=1, stress=True), pkg.weights.g_layout(C, H, W, nd))
    rng = np.random.default_rng(7)
    z = rng.normal(size=(3, nd)).astype(np.float32)
    x = rng.random(size=(3, C, H, W)).astype(np.float32)
    want, f = torch_grad.autograd_grad(p, C, H, W, nd, z, x, prior, dtype=torch.float64)
    got = torch_grad.adjoint_grad(p, C, H, W, nd, z, x, prior, dtype=torch.float64)
    assert np.abs(want).max() > 1.0, "stress weights should give an O(1)+ gradient"
    err = np.abs(got - want).max() / np.abs(want).max()
    assert err <= 1e-5, err
    assert np.isfinite(f).all() and (f > 0).all()

"""The masked objective of face completion (ganrev_refine_masked_l2; tests/masked_grad.py): the closed-form gradient with
e3 = [m] e3 equals autograd through G3, an all-ones mask is exactly the unmasked objective, and what x holds under m = 0 changes
nothing, not even NaN or Inf.  Also the host-side pieces of apply_r's completion mode (masks, grid)."""
import numpy as np
import pytest

import masked_grad as mg
from oracle import torch_grad as tg
from util import grad_floor

# + the non-square 256-wide / 256-tall shapes and the Linear^T tilings of nd 1, 300 and 4096 (about 2 s of fp64 autograd each)
GEOMS = [(1, 16, 16, 32), (1, 32, 32, 100), (3, 64, 64, 64), (1, 16, 256, 32), (3, 256, 16, 32), (1, 32, 32, 300), (1, 16, 16, 1),
         (1, 16, 16, 4096)]
GID = lambda g: "C%dx%dx%d_nd%d" % g


def block_mask(N, C, H, W):
    """A centred H/2 x W/2 hole in every channel."""
    m = np.ones((N, C, H, W), np.uint8)
    m[:, :, H // 4:H // 4 + H // 2, W // 4:W // 4 + W // 2] = 0
    return m


def random_mask(N, C, H, W, seed=3):
    return (np.random.default_rng(seed).random((N, C, H, W)) >= 0.5).astype(np.uint8)


MASKS = {"block": block_mask, "random": random_mask}


def _setup(pkg, geom, seed=7):
    C, H, W, nd = geom
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=1, stress=True), pkg.weights.g_layout(C, H, W, nd))
    rng = np.random.default_rng(seed)
    z = rng.normal(size=(3, nd)).astype(np.float32)
    x = rng.random(size=(3, C, H, W)).astype(np.float32)
    return p, z, x


@pytest.mark.parametrize("kind", sorted(MASKS))
@pytest.mark.parametrize("geom", GEOMS, ids=GID)
def test_masked_adjoint_matches_autograd(pkg, geom, kind):
    import torch
    C, H, W, nd = geom
    p, z, x = _setup(pkg, geom)
    m = MASKS[kind](3, C, H, W)
    prior = 0.05
    want, f = mg.autograd_grad(p, C, H, W, nd, z, x, prior, dtype=torch.float64, mask=m)
    got = mg.adjoint_grad(p, C, H, W, nd, z, x, prior, mask=m)
    assert np.abs(want).max() > grad_floor(nd), "stress weights should give an O(1 / sqrt(nd))+ gradient"
    err = np.abs(got - want).max() / np.abs(want).max()
    assert err <= 1e-5, err
    # the mask matters: the unmasked gradient is a different vector
    full = tg.adjoint_grad(p, C, H, W, nd, z, x, prior)
    assert np.abs(full - got).max() > 1e-3 * np.abs(got).max()
    # f is the sum over the kept pixels only
    with torch.no_grad():
        y = tg.forward_G(p, C, H, W, nd, torch.from_numpy(z).double(), torch.float64)[0].numpy()
    f_want = (np.where(m != 0, y - x, 0.0) ** 2).reshape(3, -1).sum(1) + prior * (z.astype(np.float64) ** 2).sum(1)
    assert np.allclose(f, f_want, rtol=1e-12, atol=0)


@pytest.mark.parametrize("geom", [(1, 16, 16, 32), (3, 32, 16, 24)], ids=GID)
def test_all_ones_mask_is_the_unmasked_objective(pkg, geom):
    """Bit for bit, in fp32 and fp64: objective, autograd_grad, adjoint_grad and ref_e2 (float32 and exact e3)."""
    import torch
    C, H, W, nd = geom
    p, z, x = _setup(pkg, geom, seed=8)
    ones = np.ones_like(x, np.uint8)
    for dt in (torch.float32, torch.float64):
        g0, f0 = tg.autograd_grad(p, C, H, W, nd, z, x, 0.05, dtype=dt)
        g1, f1 = mg.autograd_grad(p, C, H, W, nd, z, x, 0.05, dtype=dt, mask=ones)
        assert (g0 == g1).all() and (f0 == f1).all(), dt
    assert (tg.adjoint_grad(p, C, H, W, nd, z, x, 0.05) == mg.adjoint_grad(p, C, H, W, nd, z, x, 0.05, mask=ones)).all()
    with torch.no_grad():
        y, _, _, h2 = (t.numpy() for t in tg.forward_G(p, C, H, W, nd, torch.from_numpy(z), torch.float32))
    m2 = h2.transpose(0, 2, 3, 1) > 0
    for exact in (False, True):
        a = tg.ref_e2(y, x, p["c3.w"], m2, exact=exact)
        b = mg.ref_e2(y, x, p["c3.w"], m2, exact=exact, mask=ones)
        assert (a[0] == b[0]).all() and (a[1] == b[1]).all(), exact


@pytest.mark.parametrize("fill", ["nan", "inf", "big", "random"])
def test_holes_never_matter(pkg, fill):
    """x under m = 0 replaced by NaN / +Inf / 1e30 / other random values: every masked result is bit-identical."""
    import torch
    geom = (1, 16, 16, 32)
    C, H, W, nd = geom
    p, z, x = _setup(pkg, geom, seed=9)
    m = block_mask(3, C, H, W) & random_mask(3, C, H, W, seed=4)
    hole_vals = {"nan": np.nan, "inf": np.inf, "big": 1e30,
                 "random": np.random.default_rng(5).normal(size=x.shape).astype(np.float32) * 7}[fill]
    x2 = np.where(m != 0, x, hole_vals).astype(np.float32)
    assert not np.array_equal(x2, x, equal_nan=True)
    for dt in (torch.float32, torch.float64):
        g0, f0 = mg.autograd_grad(p, C, H, W, nd, z, x, 0.05, dtype=dt, mask=m)
        g1, f1 = mg.autograd_grad(p, C, H, W, nd, z, x2, 0.05, dtype=dt, mask=m)
        assert np.isfinite(g1).all() and np.isfinite(f1).all()
        assert (g0 == g1).all() and (f0 == f1).all(), dt
    a = mg.adjoint_grad(p, C, H, W, nd, z, x, 0.05, mask=m)
    b = mg.adjoint_grad(p, C, H, W, nd, z, x2, 0.05, mask=m)
    assert np.isfinite(b).all() and (a == b).all()
    with torch.no_grad():
        y, _, _, h2 = (t.numpy() for t in tg.forward_G(p, C, H, W, nd, torch.from_numpy(z), torch.float32))
    m2 = h2.transpose(0, 2, 3, 1) > 0
    for exact in (False, True):
        r0 = mg.ref_e2(y, x, p["c3.w"], m2, exact=exact, mask=m)
        r1 = mg.ref_e2(y, x2, p["c3.w"], m2, exact=exact, mask=m)
        assert np.isfinite(r1[0]).all() and (r0[0] == r1[0]).all() and (r0[1] == r1[1]).all(), exact


def test_masked_ref_e2_zero_inside_holes(pkg):
    """ref_e2 with a mask: +0 (value and sum of |products|) wherever every neighbour's e3 is masked, i.e. inside a hole at least
    one pixel from its edge -- the property the GPU test checks the kernel against."""
    import torch
    geom = (3, 32, 32, 24)
    C, H, W, nd = geom
    p, z, x = _setup(pkg, geom, seed=10)
    m = block_mask(3, C, H, W)
    with torch.no_grad():
        y, _, _, h2 = (t.numpy() for t in tg.forward_G(p, C, H, W, nd, torch.from_numpy(z), torch.float32))
    m2 = np.ones((3, H, W, 128), bool)
    val, tot = mg.ref_e2(y, x, p["c3.w"], m2, mask=m)
    inner = np.zeros((H, W), bool)
    inner[H // 4 + 1:H // 4 + H // 2 - 1, W // 4 + 1:W // 4 + W // 2 - 1] = True
    assert (val[:, inner] == 0).all() and (tot[:, inner] == 0).all()
    assert (np.abs(val[:, ~inner]).max(axis=-1) > 0).mean() > 0.99


def test_completion_masks_and_grid(pkg):
    m = pkg.apply_r.completionMasks((10, 1, 32, 32), seed=1)
    assert m.dtype == np.uint8 and set(np.unique(m)) == {0, 1}
    assert (m[:5, :, 8:24, 8:24] == 0).all() and m[:5].sum() == 5 * (32 * 32 - 16 * 16)
    assert abs(m[5:].mean() - 0.5) < 0.05
    assert (pkg.apply_r.completionMasks((10, 1, 32, 32), seed=1) == m).all()
    rng = np.random.default_rng(1)
    cols = [rng.random((6, 1, 8, 8)).astype(np.float32) for _ in range(5)]
    g = pkg.present.completionGrid(cols, "y")
    assert g.shape == (3, 2 * 10, 4 * (5 * 8 + 2))
    # face 0, column 3 sits at x = 1 + 3 * 8 inside the first strip, grey (y) lifted to three equal channels
    assert np.allclose(g[:, 1:9, 1 + 24:1 + 32], np.clip(cols[3][0, 0], 0, 1)[None])
    assert (g[2, 0, :] == 1.0).all() and (g[0, 0, :] == 0.0).all()       # blue border

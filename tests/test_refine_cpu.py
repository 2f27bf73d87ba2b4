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


@pytest.mark.parametrize("geom", [(1, 16, 16, 20), (3, 32, 16, 24)], ids=lambda g: "C%dx%dx%d_nd%d" % g)
def test_stage_references_compose_to_adjoint(pkg, geom):
    """The per-stage references (tests/test_gpu_refine_stages.py) chained in fp64, without the library's bf16 roundings, are the
    closed-form gradient: this pins their flips, transposes, NHWC order and Linear permutation before they judge a kernel."""
    import torch
    C, H, W, nd = geom
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=1, stress=True), pkg.weights.g_layout(C, H, W, nd))
    rng = np.random.default_rng(8)
    z = rng.normal(size=(3, nd)).astype(np.float32)
    x = rng.random(size=(3, C, H, W)).astype(np.float32)
    prior = 0.05
    with torch.no_grad():
        y, h0, h1, h2 = (t.numpy() for t in torch_grad.forward_G(p, C, H, W, nd, torch.from_numpy(z).double(), torch.float64))
    nhwc = lambda a: a.transpose(0, 2, 3, 1)
    e2, _ = torch_grad.ref_e2(y, x, p["c3.w"], nhwc(h2) > 0, exact=True)
    e1, _ = torch_grad.ref_masksum(e2, torch_grad.conv_t_weights(p, "c2", rounded=False), nhwc(h1) > 0)
    e0, _ = torch_grad.ref_masksum(e1, torch_grad.conv_t_weights(p, "c1", rounded=False), nhwc(h0) > 0)
    glin, tot = torch_grad.ref_glin(e0.reshape(3, -1), torch_grad.linear_t_weights(p, H, W, nd, rounded=False))
    got = glin + 2.0 * prior * z.astype(np.float64)
    want = torch_grad.adjoint_grad(p, C, H, W, nd, z, x, prior)
    assert np.abs(want).max() > 1.0
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max(), np.abs(got - want).max()
    assert (tot >= np.abs(glin)).all()


def test_bf16_helpers_match_torch():
    """bf16_rne (fp64 -> nearest bf16, ties to even) and f2bf (the library's host rounding) against torch's float32 -> bfloat16,
    on random values and on exact ties in both directions."""
    import torch
    rng = np.random.default_rng(9)
    v = (rng.normal(size=20000) * np.exp2(rng.integers(-30, 30, size=20000))).astype(np.float32)
    mant = rng.integers(0, 1 << 7, size=4000).astype(np.uint32)
    ties = (mant << 16) | 0x8000 | (rng.integers(100, 150, size=4000).astype(np.uint32) << 23)   # halfway between two bf16
    ties = np.concatenate([ties, ties | 0x80000000]).view(np.float32)
    assert (ties.view(np.uint32) & 0xFFFF == 0x8000).all()
    for a in (v, ties, np.array([0.0, -0.0, 1.0, -3.5], np.float32)):
        want = torch.from_numpy(a).to(torch.bfloat16).float().numpy()
        assert (torch_grad.bf16_rne(a.astype(np.float64)).astype(np.float32).view(np.uint32) == want.view(np.uint32)).all()
        assert (torch_grad.bf16_to_f32(torch_grad.f2bf(a)).view(np.uint32) == want.view(np.uint32)).all()
    nan = np.array([np.nan, -np.nan], np.float32).view(np.uint32) | 1          # signalling-looking payloads stay NaN
    assert np.isnan(torch_grad.bf16_to_f32(torch_grad.f2bf(nan.view(np.float32)))).all()
    # one rounding from fp64: a value just above a tie goes up although its float32 rounding is the tie itself
    x = np.float64(1.0) + 2.0 ** -8 + 2.0 ** -40
    assert torch_grad.bf16_rne(np.array([x]))[0] == 1.0 + 2.0 ** -7
    assert torch_grad.ulp_bf16(np.array([1.0, 1.99, -2.0])).tolist() == [2.0 ** -7, 2.0 ** -7, 2.0 ** -6]


def test_reference_weight_rounding_matches_build_refine(pkg):
    """conv_t_weights / linear_t_weights (rounded) against a loop-for-loop restatement of the library's build_refine on a small blob:
    wt[(a*co + b)*9 + t] = w[(b*ci + a)*9 + 8 - t] * s[b], then f2bf; Linear^T wm[k][s*512 + c] = f2bf(lw[(c*HW0 + s)*nd + k] * s0)."""
    C, H, W, nd = 1, 16, 16, 5
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=3, stress=True), pkg.weights.g_layout(C, H, W, nd))
    f32 = np.float32
    sc = lambda bn, i: f32(p[bn + ".g"][i]) / f32(np.sqrt(f32(p[bn + ".v"][i] + f32(1e-5))))
    for layer, bn, co_f, ci_f in (("c2", "bn2", 128, 256), ("c1", "bn1", 256, 512)):
        w = p[layer + ".w"].ravel()
        ref = torch_grad.conv_t_weights(p, layer)                       # [ci][co][3][3]
        rng = np.random.default_rng(4)
        for b, a, t in zip(rng.integers(0, co_f, 300), rng.integers(0, ci_f, 300), rng.integers(0, 9, 300)):
            want = torch_grad.bf16_to_f32(torch_grad.f2bf(np.array([f32(w[(b * ci_f + a) * 9 + (8 - t)]) * sc(bn, b)], f32)))[0]
            assert ref[a, b, t // 3, t % 3] == want, (layer, a, b, t)
    hw0 = (H // 4) * (W // 4)
    lw = p["lin.w"].ravel()
    ref = torch_grad.linear_t_weights(p, H, W, nd)
    for c in range(0, 512, 37):
        for s in range(hw0):
            fo, fn = c * hw0 + s, s * 512 + c
            for k in range(nd):
                want = torch_grad.bf16_to_f32(torch_grad.f2bf(np.array([f32(lw[fo * nd + k]) * sc("bn0", fo)], f32)))[0]
                assert ref[fn, k] == want, (c, s, k)

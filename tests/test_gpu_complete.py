"""Face completion (ganrev_refine_masked_l2): refinement of noise vectors against the known pixels only.  The masked kernels
(g_conv3_adjoint_kernel<C, true>, l2_pairs_kernel<true>) against the unmasked ones with an all-ones mask, against fp64 references
(tests/masked_grad.py, on oracle/torch_grad.py) stage by stage and against fp32 autograd end to end; holes that hold NaN / Inf / anything;
an all-zero mask; the masked distance; determinism; the resident contract; and that it completes faces better than the unmasked
refinement of zero-filled holes."""
import numpy as np
import pytest

import masked_grad as mg
from oracle import torch_grad as tg
from util import assert_bitexact, rel_l2, row_cosine

pytestmark = pytest.mark.gpu

# test_gpu_refine_stages.py's bounds; p and b over the elements with a non-zero reference (holes make many trivially exact zeros)
C_BOUND = {"e2": 2e-7, "e1": 2e-7, "e0": 2e-7, "glin": 3e-5}
P_MIN = 0.998
B_MAX = 0.02


def _glin_bound(K):
    """test_gpu_refine_stages.py's: Linear^T's error grows linearly with K = F."""
    return max(C_BOUND["glin"], 4e-10 * K)

# test_gpu_refine.py's gradient bounds (C = 1: the forward pass's bf16 rounding moves the exact gradient)
COS_TOL, REL_TOL = 0.999, 3e-2
COS_TOL_C1, REL_TOL_C1 = 0.996, 8e-2
# median RMS error on the hidden pixels, 0 over 200 iterations: first B200 run (1000 W) 47.5 with the centre hole
# (0.146 -> 0.00307) and 48.1 with 50 % dropout (0.142 -> 0.00294), halved.  Unmasked refine_l2 on the zero-filled holes ends at
# 0.300 / 0.199.
COMPLETE_FACTOR = 23.0

STAGE_GEOMS = [(1, 16, 16, 32, 5), (1, 32, 32, 100, 3), (1, 64, 64, 64, 2), (3, 64, 64, 100, 2), (3, 32, 32, 256, 3),
               (1, 16, 64, 20, 3), (3, 64, 16, 64, 3), (1, 128, 128, 32, 2), (3, 256, 256, 32, 2), (1, 16, 256, 32, 3),
               (1, 32, 32, 300, 3)]
GID = lambda g: "C%dx%dx%d_nd%d_N%d" % g
STATS = {}


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()
    for k, v in sorted(STATS.items()):
        print("masked stage stats", k, v)


def _load(pkg, ctx, C, H, W, nd, cta_pairs=0x1F, chunk=0):
    ctx.set_option("chunk", chunk)
    ctx.set_option("cta_pairs", cta_pairs)
    ctx.set_option("fuse_conv3", 0)
    try:
        gb = pkg.weights.init_G(C, H, W, nd, seed=1, stress=True)
        ctx.load_G(C, H, W, nd, gb)
    finally:
        ctx.set_option("cta_pairs", 0x1F)
        ctx.set_option("fuse_conv3", 1)
    return pkg.weights.unpack(gb, pkg.weights.g_layout(C, H, W, nd))


def _inputs(C, H, W, nd, N, seed):
    rng = np.random.default_rng(seed)
    return rng.random(size=(N, C, H, W)).astype(np.float32), rng.normal(size=(N, nd)).astype(np.float32)


def block_mask(N, C, H, W):
    """A centred H/2 x W/2 hole in every channel."""
    m = np.ones((N, C, H, W), np.uint8)
    m[:, :, H // 4:H // 4 + H // 2, W // 4:W // 4 + W // 2] = 0
    return m


def random_mask(N, C, H, W, seed=3, keep=0.5):
    return (np.random.default_rng(seed).random((N, C, H, W)) < keep).astype(np.uint8)


def _mask(kind, N, C, H, W):
    return block_mask(N, C, H, W) if kind == "block" else random_mask(N, C, H, W)


def _stages(ctx, x, m, z):
    return {s: ctx.debug_refine_masked_stage(x, m, z, s) for s in ctx.REFINE_STAGES}


def _check_bf16(key, name, got_bits, ref, tot, relu):
    """test_gpu_refine_stages.py's bf16 check; p and b over the elements whose reference is non-zero."""
    got = tg.bf16_to_f32(got_bits).astype(np.float64)
    assert (got_bits[~relu] == 0).all(), f"{key} {name}: {int((got_bits[~relu] != 0).sum())} ReLU-masked elements are not +0"
    sel = relu & (ref != 0)
    assert sel.any()
    g, r, t = got[relu], ref[relu], tot[relu]
    err = np.abs(g - r)
    u = tg.ulp_bf16(r)
    bad = err > u + C_BOUND[name] * t
    c_meas = float(np.max(np.maximum(err - u, 0.0) / np.maximum(t, 1e-300)))
    g, r = got[sel], ref[sel]
    u = tg.ulp_bf16(r)
    p_meas = float(np.mean(g == tg.bf16_rne(r)))
    b_meas = float(np.mean(np.sign(r) * (g - r) / u))
    STATS[(key, name)] = dict(c=c_meas, p=round(p_meas, 5), b=round(b_meas, 5), n=int(sel.sum()))
    assert not bad.any(), f"{key} {name}: {int(bad.sum())} outside u + c sum|terms|; worst c {c_meas:.3g}"
    assert p_meas >= P_MIN, f"{key} {name}: only {p_meas:.4f} of the non-zero elements are the correctly rounded reference"
    assert abs(b_meas) <= B_MAX, f"{key} {name}: rounding bias {b_meas:.4f} ulp"


# ---------------------------------------------------------------- 1. an all-ones mask is today's refinement, bit for bit
@pytest.mark.parametrize("geom", [(1, 32, 32, 100, 5), (3, 64, 64, 64, 3), (1, 16, 64, 20, 4), (3, 256, 256, 32, 2)], ids=GID)
def test_all_ones_mask_is_unmasked(pkg, ctx, geom):
    C, H, W, nd, N = geom
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=31)
    ones = np.ones(x.shape, np.uint8)
    kw = dict(iters=3, lr=0.02, prior=0.01)
    for u, v, what in zip(ctx.refine_masked_l2(1, x, ones, z0, **kw), ctx.refine_l2(1, x, z0, **kw), ("z", "fixed", "l2")):
        assert_bitexact(u, v, what)
    for s in ctx.REFINE_STAGES:
        assert_bitexact(ctx.debug_refine_masked_stage(x, ones, z0, s), ctx.debug_refine_stage(x, z0, s), f"stage {s}")


# ---------------------------------------------------------------- 2. the masked e2 (and what follows it) against fp64
@pytest.mark.parametrize("kind", ["block", "random"])
@pytest.mark.parametrize("geom", STAGE_GEOMS, ids=GID)
def test_masked_stages_match_fp64(pkg, ctx, geom, kind):
    C, H, W, nd, N = geom
    p = _load(pkg, ctx, C, H, W, nd)
    x, z = _inputs(C, H, W, nd, N, seed=32)
    m = _mask(kind, N, C, H, W)
    st = _stages(ctx, x, m, z)
    key = GID(geom) + "_" + kind
    m2, m1, m0 = tg.bf16_mask(st["h2"]), tg.bf16_mask(st["h1"]), tg.bf16_mask(st["h0"])
    ref, tot = mg.ref_e2(st["y"], x, p["c3.w"], m2, mask=m)
    _check_bf16(key, "e2", st["e2"], ref, tot, m2)
    # exact +0 wherever every contributing e3 is masked: no kept pixel in the 3x3 neighbourhood in any channel
    kept = np.zeros((N, H + 2, W + 2), bool)
    any_c = (m != 0).any(axis=1)
    for dy in range(3):
        for dx in range(3):
            kept[:, dy:dy + H, dx:dx + W] |= any_c
    dead = ~kept[:, 1:H + 1, 1:W + 1]
    if kind == "block":
        assert dead.sum() == N * (H // 2 - 2) * (W // 2 - 2)
    assert (st["e2"][dead] == 0).all(), f"{key}: e2 is not +0 inside the holes"
    ref, tot = tg.ref_masksum(tg.bf16_to_f32(st["e2"]), tg.conv_t_weights(p, "c2"), m1)
    _check_bf16(key, "e1", st["e1"], ref, tot, m1)
    ref, tot = tg.ref_masksum(tg.bf16_to_f32(st["e1"]), tg.conv_t_weights(p, "c1"), m0)
    _check_bf16(key, "e0", st["e0"], ref, tot, m0)
    ref, tot = tg.ref_glin(tg.bf16_to_f32(st["e0"]).reshape(N, -1), tg.linear_t_weights(p, H, W, nd))
    got = st["glin"].astype(np.float64)
    c_meas = float(np.max(np.abs(got - ref) / np.maximum(tot, 1e-300)))
    K = 512 * H * W // 16
    STATS[(key, "glin")] = dict(c=c_meas, K=K)
    assert (np.abs(got - ref) <= _glin_bound(K) * tot).all(), f"{key} glin: worst c {c_meas:.3g} at K {K}"
    # the forward half is the unmasked one
    assert_bitexact(st["y"], ctx.debug_refine_stage(x, z, "y"), "y")


def test_masked_e2_past_2g(pkg, ctx):
    """1x256x256 at chunk 264 with a block mask: element indices of h2 / e2 pass 2^31 from image 256 on.  The masked e2 of the first
    and last row of each chunk, rows 127 / 128 and rows past 2^31 / (128 H W) against fp64, and bit-identical to the same rows run
    alone.  One stage at a time, selected rows only (a stage of e2 is 4.4 GB)."""
    C, H, W, nd, N, chunk = 1, 256, 256, 32, 265, 264
    rows = np.array([0, 127, 128, 256, 263, 264])
    p = _load(pkg, ctx, C, H, W, nd, chunk=chunk)
    try:
        x, z = _inputs(C, H, W, nd, N, seed=42)
        m = block_mask(N, C, H, W)
        st = {}
        for s in ("h2", "y", "e2"):
            a = ctx.debug_refine_masked_stage(x, m, z, s)
            st[s] = a[rows].copy()
            del a
        xr, zr, mr = x[rows].copy(), z[rows].copy(), m[rows].copy()
        del x, m
        ctx.set_option("chunk", 0)
        for s in ("h2", "y", "e2"):
            assert_bitexact(ctx.debug_refine_masked_stage(xr, mr, zr, s), st[s], f"{s}: rows {rows.tolist()} alone vs inside a 264-image chunk")
    finally:
        ctx.set_option("chunk", 0)
    m2 = tg.bf16_mask(st["h2"])
    ref, tot = mg.ref_e2(st["y"], xr, p["c3.w"], m2, mask=mr)
    _check_bf16("C1x256x256_chunk264_block", "e2", st["e2"], ref, tot, m2)


# ---------------------------------------------------------------- 3. end-to-end gradient against fp32 masked autograd
@pytest.mark.parametrize("kind", ["block", "random"])
@pytest.mark.parametrize("geom", [(1, 16, 16, 32, 6), (1, 32, 32, 100, 5), (3, 64, 64, 64, 3)], ids=GID)
def test_masked_grad_matches_autograd(pkg, ctx, geom, kind):
    C, H, W, nd, N = geom
    p = _load(pkg, ctx, C, H, W, nd)
    rng = np.random.default_rng(11)
    z = rng.normal(size=(N, nd)).astype(np.float32)
    x = rng.random(size=(N, C, H, W)).astype(np.float32)
    m = _mask(kind, N, C, H, W)
    prior = np.float32(0.1)
    want, _ = mg.autograd_grad(p, C, H, W, nd, z, x, float(prior), mask=m)
    got = ctx.debug_refine_masked_stage(x, m, z, "glin") + (np.float32(2.0) * prior) * z
    cos = row_cosine(got, want)
    assert cos.min() >= (COS_TOL if C == 3 else COS_TOL_C1), cos
    assert rel_l2(got, want) <= (REL_TOL if C == 3 else REL_TOL_C1), rel_l2(got, want)


# ---------------------------------------------------------------- 4. what the holes hold never matters
@pytest.mark.parametrize("geom", [(1, 32, 32, 32, 8), (3, 64, 16, 64, 3)], ids=GID)
def test_holes_never_matter(pkg, ctx, geom):
    C, H, W, nd, N = geom
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=34)
    m = block_mask(N, C, H, W) & random_mask(N, C, H, W, seed=5, keep=0.7)
    kw = dict(iters=5, lr=0.02, prior=0.01)
    want = ctx.refine_masked_l2(1, x, m, z0, **kw)
    want_e2 = ctx.debug_refine_masked_stage(x, m, z0, "e2")
    rng = np.random.default_rng(35)
    for fill in (rng.random(x.shape).astype(np.float32) * 5 - 2, np.float32(1e30), np.float32(np.inf), np.float32(np.nan)):
        xh = np.where(m != 0, x, fill).astype(np.float32)
        got = ctx.refine_masked_l2(1, xh, m, z0, **kw)
        for u, v, what in zip(got, want, ("z", "fixed", "l2")):
            assert np.isfinite(u).all(), what
            assert_bitexact(u, v, f"{what} with holes = {fill if np.ndim(fill) == 0 else 'random'}")
        assert_bitexact(ctx.debug_refine_masked_stage(xh, m, z0, "e2"), want_e2, "e2")


# ---------------------------------------------------------------- 5. an all-zero mask; one Adam step
def _adam_np(z, g, lr, b1, b2, eps, t):
    f32 = np.float32
    m = (f32(1) - f32(b1)) * g
    v = ((f32(1) - f32(b2)) * g) * g
    step = f32(lr * np.sqrt(1.0 - float(f32(b2)) ** t) / (1.0 - float(f32(b1)) ** t))
    return z - (step * m) / (np.sqrt(v) + f32(eps))


def _ulp(a, b):
    return np.abs(a.astype(np.float32).view(np.int32).astype(np.int64) - b.astype(np.float32).view(np.int32).astype(np.int64))


def test_all_zero_mask_and_adam_step(pkg, ctx):
    C, H, W, nd, N = 1, 32, 32, 32, 40
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=36)
    zero = np.zeros(x.shape, np.uint8)
    assert (ctx.debug_refine_masked_stage(x, zero, z0, "glin") == 0).all()
    z, fixed, l2 = ctx.refine_masked_l2(1, x, zero, z0, iters=5, lr=0.05, prior=0.0)
    assert_bitexact(z, z0, "z under an all-zero mask and prior 0")
    assert (l2 == 0).all()
    assert_bitexact(fixed, ctx.forward_G(z0), "fixed")
    lr, b1, b2, eps, prior = 0.05, 0.9, 0.999, 1e-8, 0.05
    for m in (zero, random_mask(N, C, H, W, seed=6)):
        g = ctx.debug_refine_masked_stage(x, m, z0, "glin") + (np.float32(2.0) * np.float32(prior)) * z0
        z1, _, _ = ctx.refine_masked_l2(1, x, m, z0, iters=1, lr=lr, beta1=b1, beta2=b2, eps=eps, prior=prior)
        assert _ulp(z1, _adam_np(z0, g, lr, b1, b2, eps, 1)).max() <= 2
        assert np.abs(z1 - z0).max() > 0.01


# ---------------------------------------------------------------- 6. the masked distance
def test_masked_distance(pkg, ctx):
    C, H, W, nd, N = 3, 32, 32, 64, 300
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=37)
    m = random_mask(N, C, H, W, seed=7, keep=0.6)
    m[: N // 2] &= block_mask(N // 2, C, H, W)
    xh = np.where(m != 0, x, np.float32(np.nan)).astype(np.float32)
    for iters in (0, 3):
        z, fixed, l2 = ctx.refine_masked_l2(1, xh, m, z0, iters=iters, lr=0.02)
        assert_bitexact(fixed, ctx.forward_G(z), "fixed = G(z_final)")
        want = ctx.l2(np.where(m != 0, x, 0).astype(np.float32), np.where(m != 0, fixed, 0).astype(np.float32))
        assert_bitexact(l2, want, f"masked l2, iters {iters}")
        got_flags = ctx.anomaly_flags(None, N, 200, 0.15)       # the distances the call left on the device
        want_flags = ctx.anomaly_flags(want, N, 200, 0.15)
        assert (got_flags[0] == want_flags[0]).all() and got_flags[1] == want_flags[1]
    # not normalised by the kept count: l2^2 is the plain sum over the kept pixels
    d = np.where(m != 0, x.astype(np.float64) - fixed, 0.0)
    assert np.allclose(l2 ** 2, (d ** 2).reshape(N, -1).sum(1), rtol=1e-5)


# ---------------------------------------------------------------- 7. determinism, chunk independence, CTA pairs
def test_deterministic_and_chunk_independent(pkg, ctx):
    C, H, W, nd, N = 1, 32, 32, 32, 3000
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=38)
    m = random_mask(N, C, H, W, seed=8)
    m[::2] &= block_mask(1, C, H, W)
    kw = dict(iters=4, lr=0.02, prior=0.01)
    a = ctx.refine_masked_l2(1, x, m, z0, **kw)
    b = ctx.refine_masked_l2(1, x, m, z0, **kw)
    for u, v in zip(a, b):
        assert_bitexact(u, v, "repeat")
    try:
        ctx.set_option("chunk", 1000)
        c = ctx.refine_masked_l2(1, x, m, z0, **kw)
    finally:
        ctx.set_option("chunk", 0)
    for u, v in zip(a, c):
        assert_bitexact(u, v, "chunk 1000")
    for sl, what in ((slice(1000, 2000), "rows 1000-1999 alone"), (slice(0, 1), "N = 1"), (slice(0, 1337), "N = 1337")):
        d = ctx.refine_masked_l2(1, x[sl], m[sl], z0[sl], **kw)
        for u, v in zip(a, d):
            assert_bitexact(u[sl], v, what)


def test_cta_pair_matches_single_cta(pkg, ctx):
    C, H, W, nd, N = 3, 64, 16, 64, 3
    x, z = _inputs(C, H, W, nd, N, seed=39)
    m = random_mask(N, C, H, W, seed=9)
    _load(pkg, ctx, C, H, W, nd, 0x1F)
    a = _stages(ctx, x, m, z)
    _load(pkg, ctx, C, H, W, nd, 0x0F)
    b = _stages(ctx, x, m, z)
    for s in ctx.REFINE_STAGES:
        assert_bitexact(b[s], a[s], f"stage {s}: single CTA vs CTA pair")


# ---------------------------------------------------------------- 8. resident contract and errors
def test_resident_contract_and_errors(pkg, ctx):
    C, H, W, nd, N = 1, 32, 32, 32, 300
    _load(pkg, ctx, C, H, W, nd)
    ctx.load_R(1, C, H, W, nd, pkg.weights.init_R(C, H, W, nd, seed=2, stress=True))
    x, z0 = _inputs(C, H, W, nd, N, seed=40)
    m = random_mask(N, C, H, W, seed=10)
    xh = np.where(m != 0, x, np.float32(np.nan)).astype(np.float32)
    kw = dict(iters=3, lr=0.02, prior=0.01)
    zf, _, _ = ctx.fix_l2(1, xh, m)
    r = ctx.refine_masked_l2(1, None, None, None, N=N, **kw)
    s = ctx.refine_masked_l2(1, xh, m, zf, **kw)
    for u, v in zip(r, s):
        assert_bitexact(u, v, "fix_l2(1, x, m) then refine_masked_l2 on the resident buffers")
    assert_bitexact(ctx.buffer_get(pkg._lib.BUF_ATTRS1, 0, N), s[0], "ATTRS1 holds z_final")
    # iters = 0: G(z0) with the masked distance
    z_0, fixed0, l20 = ctx.refine_masked_l2(1, xh, m, z0, iters=0)
    assert_bitexact(z_0, z0, "z unchanged")
    assert_bitexact(fixed0, ctx.forward_G(z0), "G(z0)")
    assert_bitexact(l20, ctx.l2(np.where(m != 0, x, 0).astype(np.float32), np.where(m != 0, fixed0, 0).astype(np.float32)), "l2")
    for bad in (dict(iters=-1), dict(iters=1, lr=0.0), dict(iters=1, prior=-1.0)):
        with pytest.raises(pkg.GanrevError) as e:
            ctx.refine_masked_l2(1, x, m, z0, **bad)
        assert e.value.code == pkg._lib.EINVAL
    ctx.buffer_put(pkg._lib.BUF_MASK, m[:N - 1])                  # N - 1 resident mask rows
    with pytest.raises(pkg.GanrevError) as e:
        ctx.refine_masked_l2(1, x, None, z0, iters=1)
    assert e.value.code == pkg._lib.ESTATE
    try:
        ctx.set_option("conv_impl", 1)
        with pytest.raises(pkg.GanrevError) as e:
            ctx.refine_masked_l2(1, x, m, z0, iters=1)
        assert e.value.code == pkg._lib.EINVAL
    finally:
        ctx.set_option("conv_impl", 0)
    got = ctx.refine_masked_l2(1, x[:0], m[:0], z0[:0], iters=5)
    assert got[0].shape == (0, nd) and got[1].shape == (0, C, H, W) and got[2].shape == (0,)
    other = pkg.Context(0)
    try:
        other.load_R(1, C, H, W, nd, pkg.weights.init_R(C, H, W, nd, seed=2))
        with pytest.raises(pkg.GanrevError) as e:
            other.refine_masked_l2(1, x, m, z0, iters=1)
        assert e.value.code == pkg._lib.ESTATE
    finally:
        other.close()


# ---------------------------------------------------------------- 9. it completes faces
@pytest.mark.parametrize("kind", ["centre_hole", "dropout"])
def test_completes_faces(pkg, ctx, kind):
    """x = G(z*), z0 = z* + 0.5 N(0,1), pixels hidden by the mask: fitting the known pixels recovers the hidden ones, and better than
    the unmasked refinement, which fits the zero-filled holes."""
    C, H, W, nd, N = 1, 32, 32, 32, 64
    _load(pkg, ctx, C, H, W, nd)
    rng = np.random.default_rng(41)
    zs = rng.normal(size=(N, nd)).astype(np.float32)
    x = ctx.forward_G(zs)
    z0 = (zs + 0.5 * rng.normal(size=zs.shape)).astype(np.float32)
    m = block_mask(N, C, H, W) if kind == "centre_hole" else random_mask(N, C, H, W, seed=12)
    hidden = m == 0
    xh = np.where(m != 0, x, np.float32(np.nan)).astype(np.float32)

    def hidden_rms(fixed):
        return float(np.median(np.sqrt((np.where(hidden, fixed - x, 0.0) ** 2).reshape(N, -1).sum(1) / hidden.reshape(N, -1).sum(1))))

    known, rms = [], []
    for it in (0, 10, 50, 200):
        _, fixed, l2 = ctx.refine_masked_l2(1, xh, m, z0, iters=it)
        known.append(float(np.median(l2)))
        rms.append(hidden_rms(fixed))
    _, fixed_u, _ = ctx.refine_l2(1, np.where(m != 0, x, 0).astype(np.float32), z0, iters=200)
    rms_unmasked = hidden_rms(fixed_u)
    print(f"{kind}: median known-pixel l2 at 0/10/50/200 iterations {known}; median hidden RMS {rms}, factor {rms[0] / rms[-1]:.2f}; "
          f"unmasked refine_l2 on zero-filled holes: hidden RMS {rms_unmasked:.4g}")
    assert all(b <= a for a, b in zip(known, known[1:])), known
    assert rms[0] / rms[-1] >= COMPLETE_FACTOR, rms
    assert rms[-1] < rms_unmasked, (rms[-1], rms_unmasked)

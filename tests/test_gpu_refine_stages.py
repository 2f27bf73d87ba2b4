"""Refinement's backward kernels one stage at a time (ganrev_debug_refine_stage) against fp64 references of that kernel alone
(oracle/torch_grad.py), fed the library's own input to the stage: g_conv3_adjoint_kernel (e2), the MASKSUM convs conv2^T (e1) and
conv1^T (e0) in every variant, Linear^T (glin) at NT 32...256 and with up to 16 column tiles.  Also: square and non-square
geometries up to 256x256, several chunks with a ragged last one, chunks whose byte offsets (3x256x256, 256 images) and element
indices (1x256x256, 264 images) pass 2^31, refine_l2 end to end at 3x256x256, CTA pairs against single CTAs, multi-step Adam bit
for bit, and the resident contract of slot 0.

Bounds for a bf16 stage, u = the bf16 spacing at the reference:
  * every element whose stored ReLU mask is off is exactly +0;
  * |got - ref| <= u + c * sum|products|  (c: fp32 / tensor-core accumulation order);
  * got == bf16(ref) for at least a fraction p of the unmasked elements, and |mean(sign(ref) (got - ref) / u)| <= b.  The last two
    catch a biased rounding (truncation stays within one ulp everywhere); the sign makes truncation toward zero, which is
    symmetric in (got - ref), show as a mean of about -1/2.
"""
import math

import numpy as np
import pytest

from oracle import torch_grad as tg
from util import assert_bitexact

pytestmark = pytest.mark.gpu

# First B200 run (1000 W), worst over the geometries up to 64x64, every variant and depth: c 1.7e-8 (e2), 3.1e-8 (e1), 4.5e-8 (e0),
# 5.8e-6 (glin, fp32 out: no ulp of slack, K up to 131072); p >= 0.99991 (e2), 0.99952 (e1), 0.99897 (e0); |b| <= 0.0053.  Bounds:
# c x4-6, p and b at a margin that a truncating rounding (p ~ 0.5, b ~ -0.5) cannot meet.  Up to 256x256 (DESIGN section 4.5):
# e1 / e0 keep their bounds (worst c 6.6e-8 / 7.3e-8); e2's worst reached 1.005e-7 over 20 M masked elements at 1x256x256
# (tests/test_gpu_complete.py), a cancelling sum of 9 C fp32 products whose own rounding bound is about 9 C 2^-24 = 5.4e-7 C, so e2
# now shares e1's 2e-7; glin's grows with K (_glin_bound).
C_BOUND = {"e2": 2e-7, "e1": 2e-7, "e0": 2e-7, "glin": 3e-5}
P_MIN = 0.998
B_MAX = 0.02


def _glin_bound(K):
    """c of Linear^T, which sums K = F = 512 H W / 16 products into one fp32 tensor-core accumulator: like R Linear1
    (tests/test_gpu_forward_stages.py), its error grows with K.  Worst on a B200 (1000 W): 6.3e-6 at K 131072, 3.0e-5 at 524288,
    1.7e-4 at 2097152; the bound is 4e-10 K (5x at 2097152), at least the 3e-5 asserted up to 64x64."""
    return max(C_BOUND["glin"], 4e-10 * K)

GEOMS = [(1, 16, 16, 32, 5),      # conv1^T NDY 1: two 8x8 images per M tile, odd N leaves the last tile half filled
         (1, 32, 32, 100, 3),     # default shapes; Linear^T NT 128 with padded columns
         (1, 64, 64, 64, 2),      # large halo tiles
         (3, 64, 64, 100, 2),     # the C = 3 adjoint
         (3, 32, 32, 256, 3),     # Linear^T NT 256
         (1, 16, 64, 20, 3),      # non-square: H/W swaps; a ragged NT 32 column tile
         (3, 64, 16, 64, 3),      # non-square: Win = 8 halo tiles (conv1^T input 32x8)
         (1, 128, 128, 32, 2),    # conv2^T input 128 wide, the adjoint at lgH = lgW = 7; Linear^T K = 524288
         (3, 256, 256, 32, 2),    # conv2^T input 256 wide, lgH = lgW = 8; Linear^T K = 2097152
         (1, 256, 16, 32, 3),     # tall: conv1^T input 128x8
         (1, 16, 256, 32, 3),     # wide: conv2^T input 16x256, conv1^T 8x128
         (1, 32, 32, 300, 3),     # Linear^T: two NT 256 column tiles, the second ragged (44 of 256)
         (1, 16, 16, 1, 5),       # Linear^T: one column of an NT 32 tile
         (1, 16, 16, 4096, 3)]    # Linear^T: 16 NT 256 column tiles
GID = lambda g: "C%dx%dx%d_nd%d_N%d" % g

STATS = {}


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()
    for k, v in sorted(STATS.items()):
        print("stage stats", k, v)


def _load(pkg, ctx, C, H, W, nd, cta_pairs=0x1F, chunk=0):
    """fuse_conv3 = 0: forward_G then runs the same layers as the refinement's forward, so y is bit-identical to it."""
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


def _stages(ctx, x, z, rows=None):
    """Every stage buffer; rows: keep only these rows of each (bounds host memory at large N)."""
    out = {}
    for s in ctx.REFINE_STAGES:
        a = ctx.debug_refine_stage(x, z, s)
        out[s] = a if rows is None else a[rows].copy()
        del a
    return out


def _check_bf16(key, name, got_bits, ref, tot, mask):
    got = tg.bf16_to_f32(got_bits).astype(np.float64)
    off = ~mask
    assert (got_bits[off] == 0).all(), f"{key} {name}: {int((got_bits[off] != 0).sum())} masked elements are not +0"
    assert mask.any()
    g, r, t = got[mask], ref[mask], tot[mask]
    u = tg.ulp_bf16(r)
    err = np.abs(g - r)
    c_meas = float(np.max(np.maximum(err - u, 0.0) / np.maximum(t, 1e-300)))
    p_meas = float(np.mean(g == tg.bf16_rne(r)))
    b_meas = float(np.mean(np.sign(r) * (g - r) / u))
    STATS[(key, name)] = dict(c=c_meas, p=round(p_meas, 5), b=round(b_meas, 5), n=int(mask.sum()))
    bad = err > u + C_BOUND[name] * t
    assert not bad.any(), f"{key} {name}: {int(bad.sum())} of {bad.size} outside u + c sum|terms|; worst c {c_meas:.3g}, " \
                          f"first got {g[bad][:4]} want {r[bad][:4]}"
    assert p_meas >= P_MIN, f"{key} {name}: only {p_meas:.4f} of the elements are the correctly rounded reference"
    assert abs(b_meas) <= B_MAX, f"{key} {name}: rounding bias {b_meas:.4f} ulp"


def _check_chain(key, p, geom, x, z, st):
    """The references of e2, e1, e0, glin on the library's inputs to each."""
    C, H, W, nd = geom
    m2, m1, m0 = tg.bf16_mask(st["h2"]), tg.bf16_mask(st["h1"]), tg.bf16_mask(st["h0"])
    ref, tot = tg.ref_e2(st["y"], x, p["c3.w"], m2)
    _check_bf16(key, "e2", st["e2"], ref, tot, m2)
    ref, tot = tg.ref_masksum(tg.bf16_to_f32(st["e2"]), tg.conv_t_weights(p, "c2"), m1)
    _check_bf16(key, "e1", st["e1"], ref, tot, m1)
    ref, tot = tg.ref_masksum(tg.bf16_to_f32(st["e1"]), tg.conv_t_weights(p, "c1"), m0)
    _check_bf16(key, "e0", st["e0"], ref, tot, m0)
    ref, tot = tg.ref_glin(tg.bf16_to_f32(st["e0"]).reshape(len(z), -1), tg.linear_t_weights(p, H, W, nd))
    got = st["glin"].astype(np.float64)
    c_meas = float(np.max(np.abs(got - ref) / np.maximum(tot, 1e-300)))
    K = 512 * H * W // 16
    STATS[(key, "glin")] = dict(c=c_meas, K=K)
    assert (np.abs(got - ref) <= _glin_bound(K) * tot).all(), f"{key} glin: worst c {c_meas:.3g} at K {K}"


@pytest.mark.parametrize("cta_pairs", [0x1F, 0], ids=["pairs", "single"])
@pytest.mark.parametrize("geom", GEOMS, ids=GID)
def test_stages_match_fp64(pkg, ctx, geom, cta_pairs):
    C, H, W, nd, N = geom
    p = _load(pkg, ctx, C, H, W, nd, cta_pairs)
    x, z = _inputs(C, H, W, nd, N, seed=21)
    st = _stages(ctx, x, z)
    # y: the forward half of the grad chunk is forward_G itself (same layers, same gather), and forward_G is G
    assert_bitexact(st["y"], ctx.forward_G(z), "y = forward_G(z)")
    import torch
    with torch.no_grad():
        y64 = tg.forward_G(p, C, H, W, nd, torch.from_numpy(z).double(), torch.float64)[0].numpy()
    assert np.abs(st["y"] - y64).max() <= 2e-2, np.abs(st["y"] - y64).max()        # the smoke test's bound for G's pixels
    _check_chain(GID(geom) + ("" if cta_pairs else "_single"), p, (C, H, W, nd), x, z, st)
    # the hook is the gradient the optimiser sees: glin + 2 prior z is debug_refine_grad bit for bit
    prior = np.float32(0.1)
    grad, _ = ctx.debug_refine_grad(x, z, float(prior))
    assert_bitexact(st["glin"] + (np.float32(2.0) * prior) * z, grad, "glin + 2 prior z")


@pytest.mark.parametrize("geom", [(1, 32, 32, 100, 1100), (1, 16, 16, 32, 1101)], ids=GID)
def test_stages_deep(pkg, ctx, geom):
    """chunk 512: two full chunks and a ragged third, ~14 conv2^T work items per persistent CTA.  References on 16 rows: the first
    and last row of every chunk and random rows."""
    C, H, W, nd, N = geom
    p = _load(pkg, ctx, C, H, W, nd, chunk=512)
    try:
        x, z = _inputs(C, H, W, nd, N, seed=22)
        rng = np.random.default_rng(23)
        edges = [0, 511, 512, 1023, 1024, N - 1]
        rest = np.setdiff1d(np.arange(N), edges)
        rows = np.sort(np.concatenate([edges, rng.choice(rest, 16 - len(edges), replace=False)]))
        st = _stages(ctx, x, z, rows)
        _check_chain(GID(geom), p, (C, H, W, nd), x[rows], z[rows], st)
        # and the same rows alone, in one chunk
        ctx.set_option("chunk", 0)
        alone = _stages(ctx, x[rows], z[rows])
        for s in ctx.REFINE_STAGES:
            assert_bitexact(alone[s], st[s], f"stage {s}: rows alone vs inside three chunks")
    finally:
        ctx.set_option("chunk", 0)


# (C, H, W, nd, N, chunk): 3x256x256 at the default chunk (256 images): h2 / e2 of a full chunk are 2^31 bf16 elements, byte offsets
# pass 2^31 from image 128 on, and a ragged one-image chunk follows.  1x256x256 at chunk 264: element indices of h2 / e2 (and of G's
# conv2 output in forward_G) pass 2^31 from image 256 on, 2^31 / (128 H W) = 256.
PAST_2G = [(3, 256, 256, 32, 257, 0), (1, 256, 256, 32, 265, 264)]
PID = lambda g: "C%dx%dx%d_nd%d_N%d_chunk%d" % g


def past_2g_rows(N, chunk):
    """First and last row of each chunk, rows 127 / 128 (byte offsets pass 2^31 at 128) and rows past element index 2^31."""
    CH = chunk or 256
    rows = {127, 128, 256, N - 1}
    for n0 in range(0, N, CH):
        rows |= {n0, min(n0 + CH, N) - 1}
    return np.array(sorted(rows))


@pytest.mark.parametrize("geom", PAST_2G, ids=PID)
def test_full_chunk_past_2g(pkg, ctx, geom):
    """Every stage on the selected rows against fp64, and bit-identical to the same rows run alone (one small chunk); y is
    forward_G's.  One stage is fetched at a time and only its selected rows are kept: a stage of e2 is 4.4 GB at N = 265."""
    C, H, W, nd, N, chunk = geom
    rows = past_2g_rows(N, chunk)
    p = _load(pkg, ctx, C, H, W, nd, chunk=chunk)
    try:
        x, z = _inputs(C, H, W, nd, N, seed=29)
        st = _stages(ctx, x, z, rows)
        assert_bitexact(st["y"], ctx.forward_G(z)[rows], "y = forward_G(z), rows")
        xr, zr = x[rows].copy(), z[rows].copy()
        del x
        ctx.set_option("chunk", 0)
        alone = _stages(ctx, xr, zr)
    finally:
        ctx.set_option("chunk", 0)
    for s in ctx.REFINE_STAGES:
        assert_bitexact(alone[s], st[s], f"stage {s}: rows {rows.tolist()} alone vs inside chunks of {chunk or 256}")
    import torch
    with torch.no_grad():
        y64 = tg.forward_G(p, C, H, W, nd, torch.from_numpy(zr).double(), torch.float64)[0].numpy()
    assert np.abs(st["y"] - y64).max() <= 2e-2, np.abs(st["y"] - y64).max()
    _check_chain(PID(geom), p, (C, H, W, nd), xr, zr, st)


def test_refine_l2_256(pkg, ctx):
    """refine_l2 end to end at 3x256x256 over a full chunk and a ragged one: the checked rows' z is what refining them alone gives,
    fixed is forward_G(z) and l2 is ctx.l2(x, fixed), bit for bit."""
    C, H, W, nd, N = 3, 256, 256, 32, 257
    rows = past_2g_rows(N, 0)
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=30)
    kw = dict(iters=2, lr=0.02, prior=0.01)
    z, fixed, l2 = ctx.refine_l2(1, x, z0, **kw)
    assert np.abs(z - z0).max() > 1e-3
    assert_bitexact(fixed, ctx.forward_G(z), "fixed = forward_G(z_final)")
    assert_bitexact(l2, ctx.l2(x, fixed), "l2 = ctx.l2(x, fixed)")
    del fixed
    za, _, _ = ctx.refine_l2(1, x[rows], z0[rows], want_fixed=False, **kw)
    assert_bitexact(za, z[rows], f"z of rows {rows.tolist()} refined alone")


@pytest.mark.parametrize("geom", [(1, 32, 32, 100, 4), (3, 64, 16, 64, 3)], ids=GID)
def test_cta_pair_matches_single_cta(pkg, ctx, geom):
    """cta_pairs bit 4 selects conv2^T / conv1^T as CTA pairs (NDY 3, CG 2) or single CTAs (CG 1); the forward layers are the same
    in both.  Each accumulator sums K in the same order either way: the results are bit-identical (measured on a B200)."""
    C, H, W, nd, N = geom
    x, z = _inputs(C, H, W, nd, N, seed=24)
    _load(pkg, ctx, C, H, W, nd, 0x1F)
    a = _stages(ctx, x, z)
    _load(pkg, ctx, C, H, W, nd, 0x0F)
    b = _stages(ctx, x, z)
    for s in ctx.REFINE_STAGES:
        assert_bitexact(b[s], a[s], f"stage {s}: single CTA vs CTA pair")


def _adam_chain(ctx, x, z0, iters, lr, beta1, beta2, eps, prior, zclamp):
    """refine_adam_kernel restated in float32 numpy, the step size as the host computes it (float32 hyperparameters, then double
    pow / sqrt, then float), on the library's gradient at every z_t."""
    f32 = np.float32
    lr, b1, b2, eps, zc = f32(lr), f32(beta1), f32(beta2), f32(eps), f32(zclamp)
    z = z0.copy()
    m = np.zeros_like(z)
    v = np.zeros_like(z)
    for t in range(1, iters + 1):
        g, _ = ctx.debug_refine_grad(x, z, float(f32(prior)))
        step = f32(float(lr) * math.sqrt(1.0 - math.pow(float(b2), float(t))) / (1.0 - math.pow(float(b1), float(t))))
        m = b1 * m + (f32(1) - b1) * g
        v = b2 * v + ((f32(1) - b2) * g) * g
        z = z - (step * m) / (np.sqrt(v) + eps)
        if zc > 0:
            z = np.minimum(np.maximum(z, -zc), zc)
        assert z.dtype == np.float32
    return z


def test_adam_multi_step_bitexact(pkg, ctx):
    """Six steps with prior > 0, non-default beta1 / beta2 and a binding clamp, over two chunks (m / v start at zero per chunk)."""
    _adam_multi_step(pkg, ctx, 32)


def test_adam_multi_step_bitexact_nd300(pkg, ctx):
    """The same at nd 300: two Linear^T column tiles, the second ragged, and Adam's rows 300 floats apart."""
    _adam_multi_step(pkg, ctx, 300)


def _adam_multi_step(pkg, ctx, nd):
    C, H, W, N = 1, 32, 32, 100
    _load(pkg, ctx, C, H, W, nd, chunk=64)
    try:
        x, z0 = _inputs(C, H, W, nd, N, seed=26)
        hy = dict(lr=0.03, beta1=0.8, beta2=0.99, eps=1e-6, prior=0.1, zclamp=1.5)
        want = _adam_chain(ctx, x, z0, 6, **hy)
        got, _, _ = ctx.refine_l2(1, x, z0, iters=6, **hy)
        assert_bitexact(got, want, "refine_l2(iters=6) vs the numpy Adam chain")
        assert (np.abs(got) == np.float32(1.5)).any() and np.abs(got).max() <= np.float32(1.5)
        assert np.abs(got - z0).max() > 0.05
    finally:
        ctx.set_option("chunk", 0)


@pytest.mark.parametrize("with_z0", [True, False], ids=["z0", "in_place"])
def test_refine_slot0_unsets_aliasing_database(pkg, ctx, with_z0):
    C, H, W, nd, N = 1, 16, 16, 32, 40
    _load(pkg, ctx, C, H, W, nd)
    x, z0 = _inputs(C, H, W, nd, N, seed=27)
    ctx.buffer_put(pkg._lib.BUF_ATTRS0, z0)
    ctx.db_set(None, N=N, d=nd)
    ids, _ = ctx.search_cosine(z0[:2], 3)
    assert ids[:, 0].tolist() == [0, 1]
    ctx.refine_l2(0, x, z0 if with_z0 else None, iters=2, N=N)
    with pytest.raises(pkg.GanrevError) as e:
        ctx.search_cosine(z0[:2], 3)
    assert e.value.code == pkg._lib.ESTATE


def test_stage_errors(pkg, ctx):
    C, H, W, nd, N = 1, 16, 16, 32, 2
    _load(pkg, ctx, C, H, W, nd)
    x, z = _inputs(C, H, W, nd, N, seed=28)
    for bad in (-1, 8):
        with pytest.raises(pkg.GanrevError) as e:
            ctx.debug_refine_stage(x, z, bad)
        assert e.value.code == pkg._lib.EINVAL
    out = np.empty((N, nd), np.float32)
    L = pkg._lib
    for nbytes in (out.nbytes - 4, out.nbytes + 4):
        rc = L.lib().ganrev_debug_refine_stage(ctx._h, L._ptr(x), L._ptr(z), N, 7, L._ptr(out), nbytes)
        assert rc == L.EINVAL
    assert L.lib().ganrev_debug_refine_stage(ctx._h, L._ptr(x), L._ptr(z), N, 7, L._ptr(out), out.nbytes) == L.OK

"""G's and R's forward kernels one layer at a time (ganrev_debug_G_stage / ganrev_debug_R_stage) against fp64 references of that
layer alone (oracle/torch_layers.py), fed the library's own input to the layer: G's Linear, the phase-form upsample+convs, the last
conv's tap products (fused into conv2's epilogue or a 1x1 GEMM) and the gather + sigmoid; R's conv1 (hi/lo split input, fixer
mask), the ELU convs and their pooled epilogues, both Linears (permutations, the x0.75 fold, tanh).  Square and non-square
geometries up to 256x256, every kernel variant where it is reachable, several chunks with a ragged last one, a full 256-image chunk
at 256x256 whose conv2 output passes 2^31 bytes, and bit-identity across the store / pipeline knobs.

Bounds for a bf16 stage, u = the bf16 spacing at the reference, T = the sum of |terms| (products and the folded bias):
  * |got - ref| <= u + c * T + a   (c: fp32 / tensor-core accumulation order; a: an explicit allowance for elu_fast's ex2.approx,
    ELU layers only);
  * ReLU outputs whose reference is below -c * T are exactly +0;
  * got == bf16(ref) for at least a fraction p of the elements, and |mean(sign(ref) (got - ref) / u)| <= b, both over the elements
    where u >= 8 a (and, for ReLU, the reference is above c * T), so that ELU outputs near zero do not dilute them.  Truncation
    stays within one ulp everywhere; these two catch it (p ~ 1/2, b ~ -1/2).
Pooled stages take the largest T of each 2x2 window.  fp32 stages (taps, y, out) have no ulp term; y's a covers __expf and the
division of the sigmoid.
"""
import numpy as np
import pytest

from oracle import torch_grad as tg
from oracle import torch_layers as tl
from util import assert_bitexact

pytestmark = pytest.mark.gpu
ESTATE = 4   # GANREV_ESTATE

# First B200 run (1000 W), worst over every geometry and variant below (measured / asserted, about 5x):
#   c: G.lin 8.3e-9 / 4e-8, G.c1 1.3e-7 / 6e-7, G.c2 8.6e-8 / 4e-7, G.taps 1.5e-7 / 7e-7, G.taps_fused 2.4e-8 / 1.2e-7,
#      G.y 1.2e-7 / 6e-7, R.c1 1.6e-8 / 8e-8, R.c2..c6 4.0e-8..7.3e-8 / 2e-7..3.5e-7, R.out 1.3e-7 / 6e-7 (tanh 4.5e-8).
#   a (what the ELU layers leave beyond u + c T, c measured on their positive outputs): <= 1.6e-6 / 6e-6; G.y's largest
#      error 1.5e-7 / 6e-7.
#   p >= 0.99927 / 0.998 and |b| <= 0.0034 / 0.02, R Linear1 apart.
# R Linear1 sums K = 128 H W / 16 products (8192 at 32x32, 524288 at 256x256) into one fp32 tensor-core accumulator, and its
# error grows linearly with K: c 1.4e-7 at K 32768, 5.5e-7 at 131072, 1.7e-6 at 524288 (about 3.5e-8 K / 8192), so its bound
# is 2e-11 K; p falls to 0.987 / 0.946 / 0.860 and |b| rises to 0.012 / 0.040 / 0.085 (see DESIGN section 4.6).
C_BOUND = {"G.lin": 4e-8, "G.c1": 6e-7, "G.c2": 4e-7, "G.taps": 7e-7, "G.taps_fused": 1.2e-7, "G.y": 6e-7,
           "R.c1": 8e-8, "R.c2": 2e-7, "R.c3": 3e-7, "R.c4": 3.5e-7, "R.c5": 3e-7, "R.c6": 3.5e-7, "R.out": 6e-7}
A_ACT = {"G.y": 6e-7, "R.c1": 6e-6, "R.c2": 6e-6, "R.c3": 6e-6, "R.c4": 6e-6, "R.c5": 6e-6, "R.c6": 6e-6, "R.l1": 6e-6}
P_MIN = 0.998
B_MAX = 0.02


def _l1_bounds(K):
    """(c, p, b) of R Linear1 with K = 128 H W / 16 terms per output."""
    if K <= 32768:
        return 2e-11 * K, 0.98, 0.05
    return 2e-11 * K, (0.9 if K <= 131072 else 0.75), 0.2


RELU = ("G.lin", "G.c1", "G.c2")
ELU = ("R.c1", "R.c2", "R.c3", "R.c4", "R.c5", "R.c6", "R.l1")

# (C, H, W, nd, N, fixer): fixer = R's input goes through a dropout mask (the fixer R of apply_r)
GEOMS = [(1, 16, 16, 32, 5, True),       # NDY 1 everywhere (no halo tiles); odd N leaves tiles half filled
         (1, 32, 32, 100, 4, False),     # bench.py's geometry
         (3, 32, 32, 64, 3, True),
         (3, 64, 64, 256, 2, False),     # R Linear2 NT 256
         (1, 16, 64, 20, 3, False),      # non-square; ragged NT 32 output tile
         (3, 64, 16, 64, 3, True),       # non-square: 8-wide quarter-resolution rows
         (1, 256, 16, 32, 2, True),      # tall: 64x4 Linear layouts
         (1, 128, 128, 32, 2, False)]
GID = lambda g: "C%dx%dx%d_nd%d_N%d" % g[:5] + ("_fixer" if g[5] else "")

STATS = {}


@pytest.fixture(scope="module")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()
    for k, v in sorted(STATS.items()):
        print("stage stats", k, v)


def _opts(ctx, **kw):
    for k, v in kw.items():
        ctx.set_option(k, v)


DEFAULTS = dict(chunk=0, cta_pairs=0x1F, fuse_conv3=1, conv_impl=0, tma_store=1, xpose2=1, tma_hybrid=0, pdl=0, ups_cycles=512)


def _load(pkg, ctx, C, H, W, nd, R=True, **opts):
    """Load G (seed 1) and R (seed 2, slot 0; slot 1 with tanh) with `opts` set during the load; returns (G params, R params).
    Options read at run time (chunk, conv_impl, tma_store, tma_hybrid, pdl) stay set until _reset."""
    try:
        _opts(ctx, **opts)
        gb = pkg.weights.init_G(C, H, W, nd, seed=1, stress=True)
        ctx.load_G(C, H, W, nd, gb)
        gp = pkg.weights.unpack(gb, pkg.weights.g_layout(C, H, W, nd))
        rp = None
        if R:
            rb = pkg.weights.init_R(C, H, W, nd, seed=2, stress=True)
            ctx.load_R(0, C, H, W, nd, rb)
            ctx.load_R(1, C, H, W, nd, rb, tanh_out=True)
            rp = pkg.weights.unpack(rb, pkg.weights.r_layout(C, H, W, nd))
    finally:
        for k in ("cta_pairs", "fuse_conv3", "xpose2", "ups_cycles"):   # read at load time
            ctx.set_option(k, DEFAULTS[k])
    return gp, rp


def _reset(ctx):
    _opts(ctx, **DEFAULTS)


def _inputs(C, H, W, nd, N, seed, fixer):
    rng = np.random.default_rng(seed)
    z = rng.normal(size=(N, nd)).astype(np.float32)
    x = rng.random(size=(N, C, H, W)).astype(np.float32)
    m = (rng.random(size=x.shape) >= 0.3).astype(np.uint8) if fixer else None
    return z, x, m


def _g_stages(ctx, z, rows=None):
    fused = None
    out = {}
    for s in ctx.G_STAGES:
        try:
            a = ctx.debug_G_stage(z, s)
        except Exception as e:   # c2 when the tap products are fused: GANREV_ESTATE
            assert s == "c2" and getattr(e, "code", None) == ESTATE, e
            fused = True
            continue
        out[s] = a if rows is None else a[rows].copy()
    out["fused"] = bool(fused)
    return out


def _r_stages(ctx, slot, x, mask, rows=None, stages=None):
    out = {}
    for s in stages or ctx.R_STAGES:
        a = ctx.debug_R_stage(slot, x, s, mask)
        out[s] = a if rows is None else a[rows].copy()
    return out


def _record(key, name, **kw):
    cur = STATS.setdefault((key, name), {})
    for k, v in kw.items():
        if k in ("p",):
            cur[k] = min(cur.get(k, 1.0), round(v, 5))
        elif k == "b":
            cur[k] = max(cur.get(k, 0.0), round(abs(v), 5))
        elif k == "n":
            cur[k] = cur.get(k, 0) + v
        else:
            cur[k] = max(cur.get(k, 0.0), float("%.3g" % v))


def _check_bf16(key, name, got_bits, ref, tot, pre=None, K=None):
    """One bf16 stage; ref = the activation's output, pre = its input (ReLU layers); K: R Linear1's reduction length."""
    got = tg.bf16_to_f32(got_bits).astype(np.float64)
    if name == "R.l1":
        c, p_min, b_max = _l1_bounds(K)
    else:
        c, p_min, b_max = C_BOUND[name], P_MIN, B_MAX
    a = A_ACT.get(name, 0.0)
    u = tg.ulp_bf16(ref)
    err = np.abs(got - ref)
    if name in RELU:
        off = pre < -c * tot
        assert (got_bits[off] == 0).all(), f"{key} {name}: {int((got_bits[off] != 0).sum())} ReLU outputs are not +0"
        live = pre > c * tot
        c_meas = float(np.max(np.maximum(err - u, 0.0) / np.maximum(tot, 1e-300)))
        a_meas = 0.0
    else:
        live = u >= 8 * a
        ident = ref > 0                                   # ELU is the identity there: no activation error
        c_meas = float(np.max(np.maximum(err - u, 0.0)[ident] / np.maximum(tot[ident], 1e-300))) if ident.any() else 0.0
        a_meas = float(np.max(np.maximum(err - u - c_meas * tot, 0.0)))
    assert live.mean() > 0.2, f"{key} {name}: only {live.mean():.3f} of the elements take part in the rounding statistics"
    g, r = got[live], ref[live]
    p_meas = float(np.mean(g == tg.bf16_rne(r)))
    b_meas = float(np.mean(np.sign(r) * (g - r) / tg.ulp_bf16(r)))
    _record(key, name, c=c_meas, a=a_meas, p=p_meas, b=b_meas, n=int(live.sum()))
    bad = err > u + c * tot + a
    assert not bad.any(), f"{key} {name}: {int(bad.sum())} of {bad.size} outside u + c T + a; worst c {c_meas:.3g} a {a_meas:.3g}, " \
                          f"first got {got[bad][:4]} want {ref[bad][:4]}"
    assert p_meas >= p_min, f"{key} {name}: only {p_meas:.4f} of the elements are the correctly rounded reference"
    assert abs(b_meas) <= b_max, f"{key} {name}: rounding bias {b_meas:.4f} ulp"


def _check_f32(key, name, got, ref, tot, a_name=None):
    a = A_ACT.get(a_name or name, 0.0)
    err = np.abs(got.astype(np.float64) - ref)
    c_meas = float(np.max(err / np.maximum(tot, 1e-300)))
    _record(key, a_name or name, c=c_meas, a=float(err.max()))
    bad = err > C_BOUND[name] * tot + a
    assert not bad.any(), f"{key} {a_name or name}: {int(bad.sum())} of {bad.size} outside c T + a; worst c {c_meas:.3g}, " \
                          f"first got {got[bad][:4]} want {ref[bad][:4]}"


# ---------------------------------------------------------------- per-layer checks of one set of stage buffers
class GRefs:
    """fp64 references that depend only on the inputs the library gave each layer; computed once per geometry, reused by every
    variant whose inputs are the same bits."""

    def __init__(self, gp, C, H, W, nd, rounded=True):
        self.w = tl.g_weights(gp, C, H, W, nd, rounded)
        self.C, self.H, self.W = C, H, W
        self.cache = {}

    def get(self, name, key_bits, fn):
        k = (name, key_bits.shape, hash(key_bits.tobytes()))
        if k not in self.cache:
            self.cache[k] = fn()
        return self.cache[k]


def _check_G(key, R, z, st):
    C, H, W = R.C, R.H, R.W
    pre, tot = R.get("lin", z, lambda: tl.ref_g_lin(z, *R.w["lin"], H, W, act=False))
    _check_bf16(key, "G.lin", st["lin"], tl.relu(pre), tot, pre)
    pre, tot = R.get("c1", st["lin"], lambda: tl.ref_upconv(tl.bits(st["lin"]), *R.w["c1"], act=False))
    _check_bf16(key, "G.c1", st["c1"], tl.relu(pre), tot, pre)
    pre2, tot2 = R.get("c2", st["c1"], lambda: tl.ref_upconv(tl.bits(st["c1"]), *R.w["c2"], act=False))
    if st["fused"]:
        ref, tot = tl.ref_taps_fused(pre2, tot2, R.w["w3"])
        _check_f32(key, "G.taps_fused", st["taps"], ref, tot)
    else:
        _check_bf16(key, "G.c2", st["c2"], tl.relu(pre2), tot2, pre2)
        ref, tot = tl.ref_taps_unfused(tl.bits(st["c2"]), R.w["taps"][0])
        _check_f32(key, "G.taps", st["taps"], ref, tot)
    ref, tot = tl.ref_y(st["taps"], R.w["b3"], C)
    _check_f32(key, "G.y", st["y"], ref, tot)


def _check_R(key, rw, x, mask, st, tanh=False, simt=False):
    if simt:
        ref, tot = tl.ref_r_conv1_simt(tl.conv1_input(x, mask, split=False), *rw["c1_simt"])
    else:
        ref, tot = tl.ref_r_conv1(tl.conv1_input(x, mask), *rw["c1"])
    _check_bf16(key, "R.c1", st["c1"], ref, tot)
    for i in range(2, 7):
        ref, tot = tl.ref_conv3(tl.bits(st[f"c{i - 1}"]), *rw[f"c{i}"], pool=i in (3, 6))
        _check_bf16(key, f"R.c{i}", st[f"c{i}"], ref, tot)
    ref, tot = tl.ref_r_l1(tl.bits(st["c6"]), *rw["l1"])
    _check_bf16(key, "R.l1", st["l1"], ref, tot, K=st["c6"][0].size)
    ref, tot = tl.ref_r_out(tl.bits(st["l1"]), *rw["out"], tanh=tanh)
    _check_f32(key, "R.out", st["out"], ref, tot, "R.out_tanh" if tanh else None)   # tanhf: inside c (no extra allowance needed)


# ---------------------------------------------------------------- every geometry, default variants + fuse / tanh / fixer
@pytest.mark.parametrize("geom", GEOMS, ids=GID)
def test_G_layers_match_fp64(pkg, ctx, geom):
    """Default load (fuse_conv3 1: fused at C = 1, unfused at C = 3), then the other form of the last conv's tap products
    (fuse_conv3 0 at C = 1, 2 at C = 3): Linear and conv1 are the same bits, the taps and y are checked again."""
    C, H, W, nd, N, _ = geom
    z, _, _ = _inputs(C, H, W, nd, N, 31, False)
    gp, _ = _load(pkg, ctx, C, H, W, nd, R=False)
    refs = GRefs(gp, C, H, W, nd)
    a = _g_stages(ctx, z)
    assert a["fused"] == (C == 1)
    assert_bitexact(a["y"], ctx.forward_G(z), "y = forward_G")
    _check_G(GID(geom), refs, z, a)
    _load(pkg, ctx, C, H, W, nd, R=False, fuse_conv3=0 if C == 1 else 2)
    b = _g_stages(ctx, z)
    assert b["fused"] == (C == 3)
    for s in ("lin", "c1"):
        assert_bitexact(b[s], a[s], f"{s}: fuse_conv3 does not touch it")
    assert_bitexact(b["y"], ctx.forward_G(z), "y = forward_G")
    _check_G(GID(geom) + "_refuse", refs, z, b)
    # the refinement's forward is the same layers: h0 / h1 / h2 of debug_refine_stage are lin / c1 / c2 of the unfused load
    # (refine_grad_chunk always runs conv2 unfused, whatever fuse_conv3 was at the load)
    unf = a if C == 3 else b
    x = np.random.default_rng(32).random(size=(N, C, H, W)).astype(np.float32)
    for s, h in (("lin", "h0"), ("c1", "h1"), ("c2", "h2")):
        assert_bitexact(ctx.debug_refine_stage(x, z, h), unf[s], f"debug_refine_stage {h} = debug_G_stage {s}")


@pytest.mark.parametrize("geom", GEOMS, ids=GID)
def test_R_layers_match_fp64(pkg, ctx, geom):
    """R in slot 0 (linear output) and slot 1 (tanh; every layer before it the same bits), fixer mask where the geometry says."""
    C, H, W, nd, N, fixer = geom
    _, x, mask = _inputs(C, H, W, nd, N, 33, fixer)
    _, rp = _load(pkg, ctx, C, H, W, nd)
    rw = tl.r_weights(rp, C, H, W, nd)
    st = _r_stages(ctx, 0, x, mask)
    assert_bitexact(st["out"], ctx.forward_R(0, x, mask), "out = forward_R")
    _check_R(GID(geom), rw, x, mask, st)
    th = _r_stages(ctx, 1, x, mask, stages=("l1", "out"))
    assert_bitexact(th["l1"], st["l1"], "l1 of the tanh slot")
    assert_bitexact(th["out"], ctx.forward_R(1, x, mask), "out = forward_R (tanh)")
    ref, tot = tl.ref_r_out(tl.bits(st["l1"]), *rw["out"], tanh=True)
    _check_f32(GID(geom), "R.out", th["out"], ref, tot, "R.out_tanh")


# ---------------------------------------------------------------- kernel variants
VARIANT_GEOMS = [GEOMS[0], GEOMS[1], GEOMS[4], GEOMS[5], GEOMS[3]]


@pytest.mark.parametrize("cta_pairs", [0, 0x3F], ids=["single", "mt4"])
@pytest.mark.parametrize("geom", VARIANT_GEOMS, ids=GID)
def test_cta_variants_bit_identical(pkg, ctx, geom, cta_pairs):
    """Single CTAs (cta_pairs 0) and CTA pairs with MT = 4 for R's 64-channel convs (0x3F) against the default (0x1F): every
    accumulator sums K in the same order in all three, so every stage is the same bits.  A stage that differs is also held to
    its fp64 reference, so the failure says whether it is an order change or an error."""
    C, H, W, nd, N, fixer = geom
    z, x, mask = _inputs(C, H, W, nd, N, 34, fixer)
    _load(pkg, ctx, C, H, W, nd)
    g0, r0 = _g_stages(ctx, z), _r_stages(ctx, 0, x, mask)
    gp, rp = _load(pkg, ctx, C, H, W, nd, cta_pairs=cta_pairs)
    g1, r1 = _g_stages(ctx, z), _r_stages(ctx, 0, x, mask)
    key = GID(geom) + "_cta%02x" % cta_pairs
    diff = [f"G.{s}" for s in ctx.G_STAGES if s in g0 and not np.array_equal(g0[s], g1[s])]
    diff += [f"R.{s}" for s in ctx.R_STAGES if not np.array_equal(r0[s], r1[s])]
    if diff:
        STATS[(key, "differs")] = diff
        _check_G(key, GRefs(gp, C, H, W, nd), z, g1)
        _check_R(key, tl.r_weights(rp, C, H, W, nd), x, mask, r1)
    assert not diff, f"cta_pairs {cta_pairs:#x}: {diff} differ from the default"


KNOBS = [("tma_store", 0), ("tma_store", 2), ("xpose2", 0), ("xpose2", 2), ("tma_hybrid", 1), ("pdl", 1), ("ups_cycles", 256),
         ("ups_cycles", 2048)]


@pytest.mark.parametrize("knob", KNOBS, ids=lambda k: "%s%d" % k)
@pytest.mark.parametrize("geom", [GEOMS[1], GEOMS[5]], ids=GID)
def test_store_knobs_bit_identical(pkg, ctx, geom, knob):
    """Where results are stored (TMA bulk stores, st.global, one or two transpose buffers) and how the pipeline is staged (units
    per stage, programmatic dependent launch) do not change the order in which any accumulator sums K: every stage, same bits."""
    C, H, W, nd, N, fixer = geom
    z, x, mask = _inputs(C, H, W, nd, N, 35, fixer)
    try:
        _load(pkg, ctx, C, H, W, nd, fuse_conv3=0)
        g0, r0 = _g_stages(ctx, z), _r_stages(ctx, 0, x, mask)
        _load(pkg, ctx, C, H, W, nd, fuse_conv3=0, **{knob[0]: knob[1]})
        g1, r1 = _g_stages(ctx, z), _r_stages(ctx, 0, x, mask)
    finally:
        _reset(ctx)
    for s in ctx.G_STAGES:
        assert_bitexact(g1[s], g0[s], f"G {s}: {knob}")
    for s in ctx.R_STAGES:
        assert_bitexact(r1[s], r0[s], f"R {s}: {knob}")


@pytest.mark.parametrize("geom", [GEOMS[0], GEOMS[2]], ids=GID)
def test_cuda_core_kernels_match_fp64(pkg, ctx, geom):
    """conv_impl 1: conv_simt_kernel for every G / R conv and Linear (the tap products unfused) and r_conv1_kernel (float32 input
    and weights, BN scale applied after the sum) against the same references, on their own inputs; R with tanh too."""
    C, H, W, nd, N, fixer = geom
    z, x, mask = _inputs(C, H, W, nd, N, 36, fixer)
    try:
        gp, rp = _load(pkg, ctx, C, H, W, nd, conv_impl=1)
        g, r = _g_stages(ctx, z), _r_stages(ctx, 0, x, mask)
        assert not g["fused"]
        assert_bitexact(g["y"], ctx.forward_G(z), "y = forward_G (conv_impl 1)")
        th = ctx.debug_R_stage(1, x, "out", mask)
    finally:
        _reset(ctx)
    key = GID(geom) + "_simt"
    _check_G(key, GRefs(gp, C, H, W, nd), z, g)
    rw = tl.r_weights(rp, C, H, W, nd)
    _check_R(key, rw, x, mask, r, simt=True)
    ref, tot = tl.ref_r_out(tl.bits(r["l1"]), *rw["out"], tanh=True)
    _check_f32(key, "R.out", th, ref, tot, "R.out_tanh")


@pytest.mark.parametrize("geom", [(1, 16, 16, 32, 1100, True), (3, 32, 16, 24, 1029, False)], ids=GID)
def test_layers_deep(pkg, ctx, geom):
    """chunk 512: two full chunks and a ragged third.  References on 12 rows: the first and last row of every chunk and random
    rows; the same rows run alone (one chunk) give the same bits."""
    C, H, W, nd, N, fixer = geom
    z, x, mask = _inputs(C, H, W, nd, N, 37, fixer)
    rng = np.random.default_rng(38)
    edges = [0, 511, 512, 1023, 1024, N - 1]
    rows = np.sort(np.concatenate([edges, rng.choice(np.setdiff1d(np.arange(N), edges), 12 - len(edges), replace=False)]))
    try:
        gp, rp = _load(pkg, ctx, C, H, W, nd, chunk=512)
        g, r = _g_stages(ctx, z, rows), _r_stages(ctx, 0, x, mask, rows)
        assert_bitexact(g["y"], ctx.forward_G(z)[rows], "y = forward_G, three chunks")
        assert_bitexact(r["out"], ctx.forward_R(0, x, mask)[rows], "out = forward_R, three chunks")
        ctx.set_option("chunk", 0)
        g1, r1 = _g_stages(ctx, z[rows]), _r_stages(ctx, 0, x[rows], None if mask is None else mask[rows])
    finally:
        _reset(ctx)
    for s in ctx.G_STAGES:
        if s in g:
            assert_bitexact(g1[s], g[s], f"G {s}: rows alone vs inside three chunks")
    for s in ctx.R_STAGES:
        assert_bitexact(r1[s], r[s], f"R {s}: rows alone vs inside three chunks")
    _check_G(GID(geom), GRefs(gp, C, H, W, nd), z[rows], g)
    _check_R(GID(geom), tl.r_weights(rp, C, H, W, nd), x[rows], None if mask is None else mask[rows], r)


def test_full_chunk_past_2g(pkg, ctx):
    """3x256x256, default chunk = 256 images: G's unfused conv2 output of one chunk is 2^31 bf16 elements (4 GB), byte offsets pass
    2^31 from image 128 on and image 255 ends at element 2^31 - 1; R's conv1 output is 2 GB.  forward_G / forward_R on 257 images
    (a full chunk and a ragged one): rows 0, 127, 128, 255, 256 are the bits of the same rows run alone, and those pass every
    per-layer reference."""
    C, H, W, nd, N = 3, 256, 256, 32, 257
    rows = np.array([0, 127, 128, 255, 256])
    rng = np.random.default_rng(39)
    z = rng.normal(size=(N, nd)).astype(np.float32)
    gp, rp = _load(pkg, ctx, C, H, W, nd)
    y = ctx.forward_G(z)[rows].copy()
    x = rng.random(size=(N, C, H, W)).astype(np.float32)
    out = ctx.forward_R(0, x)[rows].copy()
    assert_bitexact(ctx.forward_G(z[rows]), y, "G rows alone vs inside a full 256-image chunk")
    xr = x[rows].copy()
    del x
    assert_bitexact(ctx.forward_R(0, xr), out, "R rows alone vs inside a full 256-image chunk")
    g = _g_stages(ctx, z[rows])
    assert not g["fused"]
    _check_G("C3x256x256_rows", GRefs(gp, C, H, W, nd), z[rows], g)
    del g
    r = _r_stages(ctx, 0, xr, None)
    _check_R("C3x256x256_rows", tl.r_weights(rp, C, H, W, nd), xr, None, r)


def test_forward_launches(pkg, ctx):
    """forward_G / forward_R launch per chunk exactly the layers they always have (the stage hooks add nothing to them)."""
    C, H, W, nd, N = 1, 32, 32, 32, 700
    z, x, _ = _inputs(C, H, W, nd, N, 40, False)
    try:
        _load(pkg, ctx, C, H, W, nd, chunk=256)
        for fuse, G_names in ((1, ["g_noise_to_bf16", "g_linear", "g_conv1_up", "g_conv2_up", "g_conv3_gather"]),
                              (0, ["g_noise_to_bf16", "g_linear", "g_conv1_up", "g_conv2_up", "g_conv3_taps", "g_conv3_gather"])):
            _load(pkg, ctx, C, H, W, nd, fuse_conv3=fuse)
            ctx.profile_reset()
            ctx.profile_enable(True)
            ctx.forward_G(z)
            ctx.forward_R(0, x)
            prof = ctx.profile()
            ctx.profile_enable(False)
            R_names = ["r_conv1", "r_conv2", "r_conv3_pool", "r_conv4", "r_conv5", "r_conv6_pool", "r_linear1", "r_linear2"]
            assert sorted(prof) == sorted(G_names + R_names), sorted(prof)
            assert all(prof[k]["launches"] == 3 for k in prof), {k: prof[k]["launches"] for k in prof}
    finally:
        ctx.profile_enable(False)
        _reset(ctx)


def test_stage_errors(pkg, ctx):
    C, H, W, nd, N = 1, 16, 16, 32, 2
    z, x, _ = _inputs(C, H, W, nd, N, 41, False)
    L = pkg._lib
    _load(pkg, ctx, C, H, W, nd)
    for bad in (-1, 5):
        with pytest.raises(pkg.GanrevError) as e:
            ctx.debug_G_stage(z, bad)
        assert e.value.code == L.EINVAL
    for bad in (-1, 8):
        with pytest.raises(pkg.GanrevError) as e:
            ctx.debug_R_stage(0, x, bad)
        assert e.value.code == L.EINVAL
    with pytest.raises(pkg.GanrevError) as e:
        ctx.debug_G_stage(z, "c2")                      # fused at C = 1: h2 never exists
    assert e.value.code == L.ESTATE
    y = np.empty((N, C, H, W), np.float32)
    for nbytes in (y.nbytes - 4, y.nbytes + 4):
        assert L.lib().ganrev_debug_G_stage(ctx._h, L._ptr(z), N, 4, L._ptr(y), nbytes) == L.EINVAL
    assert L.lib().ganrev_debug_G_stage(ctx._h, L._ptr(z), N, 4, L._ptr(y), y.nbytes) == L.OK
    o = np.empty((N, nd), np.float32)
    assert L.lib().ganrev_debug_R_stage(ctx._h, 0, L._ptr(x), None, N, 7, L._ptr(o), o.nbytes - 4) == L.EINVAL
    assert L.lib().ganrev_debug_R_stage(ctx._h, 2, L._ptr(x), None, N, 7, L._ptr(o), o.nbytes) == L.EINVAL
    assert L.lib().ganrev_debug_R_stage(ctx._h, 0, L._ptr(x), None, N, 7, L._ptr(o), o.nbytes) == L.OK

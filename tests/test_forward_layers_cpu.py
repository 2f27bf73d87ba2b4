"""The per-layer forward references (oracle/torch_layers.py) that judge G's and R's kernels in tests/test_gpu_forward_stages.py:
chained in fp64 without the library's roundings they are G and R themselves (oracle/torch_cpu.py run in fp64), which pins their
conventions (phase taps, NHWC orders, permutations, the x0.75 fold, the gather's tap planes); and each weight rounding is a
loop-by-loop restatement of load_G_impl / load_R_impl / build_tc_layer."""
import numpy as np
import pytest

from oracle import torch_layers as tl

GEOMS = [(1, 16, 16, 20), (3, 32, 16, 24), (1, 16, 32, 8)]
GID = lambda g: "C%dx%dx%d_nd%d" % g


def _double(net):
    net.p = {k: v.double() for k, v in net.p.items()}
    return net


@pytest.mark.parametrize("geom", GEOMS, ids=GID)
def test_G_references_compose_to_G(pkg, geom):
    import torch
    from oracle import torch_cpu
    C, H, W, nd = geom
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=1, stress=True), pkg.weights.g_layout(C, H, W, nd))
    z = np.random.default_rng(5).normal(size=(3, nd)).astype(np.float32)
    gw = tl.g_weights(p, C, H, W, nd, rounded=False)
    h0, t0 = tl.ref_g_lin(z, *gw["lin"], H, W, rounded=False)
    h1, t1 = tl.ref_upconv(h0, *gw["c1"])
    pre2, t2 = tl.ref_upconv(h1, *gw["c2"], act=False)
    taps_f, tf = tl.ref_taps_fused(pre2, t2, gw["w3"])
    taps_u, tu = tl.ref_taps_unfused(tl.relu(pre2), gw["taps"][0])
    y, ty = tl.ref_y(taps_f, gw["b3"], C)
    with torch.no_grad():
        want = _double(torch_cpu.TorchG(p, C, H, W, nd))(torch.from_numpy(z).double()).numpy()
    assert np.abs(want - 0.5).max() > 0.3, "stress weights should drive the sigmoid well away from 1/2"
    assert np.abs(y - want).max() <= 1e-12, np.abs(y - want).max()
    assert np.abs(taps_u - taps_f).max() <= 1e-12 * np.abs(taps_f).max()
    for v, t in ((h0, t0), (h1, t1), (pre2, t2), (taps_f, tf), (taps_u, tu)):
        assert (t >= np.abs(v) * (1 - 1e-12)).all()
    assert (ty >= 0).all() and (tu <= tf * (1 + 1e-12)).all()


@pytest.mark.parametrize("tanh", [False, True], ids=["linear", "tanh"])
@pytest.mark.parametrize("fixer", [False, True], ids=["plain", "fixer"])
@pytest.mark.parametrize("geom", GEOMS, ids=GID)
def test_R_references_compose_to_R(pkg, geom, fixer, tanh):
    import torch
    from oracle import torch_cpu
    C, H, W, nd = geom
    p = pkg.weights.unpack(pkg.weights.init_R(C, H, W, nd, seed=2, stress=True), pkg.weights.r_layout(C, H, W, nd))
    rng = np.random.default_rng(6)
    x = rng.random(size=(3, C, H, W)).astype(np.float32)
    mask = (rng.random(size=x.shape) >= 0.5).astype(np.uint8) if fixer else None
    rw = tl.r_weights(p, C, H, W, nd, rounded=False)
    a, _ = tl.ref_r_conv1(tl.conv1_input(x, mask, split=False), *rw["c1"])
    b, _ = tl.ref_r_conv1_simt(tl.conv1_input(x, mask, split=False), *rw["c1_simt"])
    assert np.abs(a - b).max() <= 1e-12
    for i in range(2, 7):
        a, t = tl.ref_conv3(a, *rw[f"c{i}"], pool=i in (3, 6))
        assert (t >= np.abs(a) * (1 - 1e-12)).all()
    a, _ = tl.ref_r_l1(a, *rw["l1"])
    got, tot = tl.ref_r_out(a, *rw["out"], tanh=tanh)
    xin = torch.from_numpy(x).double() * (torch.from_numpy(mask).double() if fixer else 1.0)
    with torch.no_grad():
        want = _double(torch_cpu.TorchR(p, C, H, W, nd))(xin)
        want = (torch.tanh(want) if tanh else want).numpy()
    assert np.abs(want).max() > 0.1
    assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), np.abs(got - want).max()


def test_conv1_input_split():
    """hi + lo is x to 2^-16 relative; hi is x's top 16 bits; lo is truncated toward zero; masked taps are 0."""
    rng = np.random.default_rng(7)
    x = (rng.normal(size=4096) * np.exp2(rng.integers(-10, 10, size=4096))).astype(np.float32)
    s = tl.conv1_input(x)
    assert (np.abs(s - x) <= np.abs(x.astype(np.float64)) * 2.0 ** -15).all()
    hi = (x.view(np.uint32) & 0xFFFF0000).view(np.float32).astype(np.float64)
    lo = x.astype(np.float64) - hi
    assert (np.abs(s - hi) <= np.abs(lo)).all() and (np.sign(s - hi) * np.sign(lo) >= 0).all()
    assert (tl.conv1_input(np.float32([1.0 + 2.0 ** -20, 3.0])) == [1.0 + 2.0 ** -20, 3.0]).all()   # both halves exact here
    m = np.array([1, 0, 2], np.uint8)
    assert tl.conv1_input(np.float32([1.5, 2.5, 3.5]), m).tolist() == [1.5, 0.0, 3.5]


def _f2bf(v):
    return float(tl.bf(np.array([v], np.float32))[0])


def test_G_weight_rounding_matches_load_G(pkg):
    """Loop-by-loop restatement of load_G_impl: Linear wm[fn = s*512 + c][k] = f2bf(lw[fo = c*HW0 + s][k] * scale[fn]); the phase
    filters wb[ph][co][(gi*ndy + j)*Cin + ci] = f2bf(float(sum * scale[co])) over S[a][ty] x S[b][tx]; tap GEMM rows t*C + co."""
    C, H, W, nd = 3, 16, 32, 5
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=3, stress=True), pkg.weights.g_layout(C, H, W, nd))
    gw = tl.g_weights(p, C, H, W, nd)
    f32 = np.float32

    def fold(bias, bn, i):
        s = f32(p[bn + ".g"][i]) / f32(np.sqrt(f32(p[bn + ".v"][i] + f32(1e-5))))
        return s, f32(p[bn + ".b"][i] + f32(f32(bias[i]) - f32(p[bn + ".m"][i])) * s)

    hw0 = (H // 4) * (W // 4)
    rng = np.random.default_rng(4)
    for c, s, k in zip(rng.integers(0, 512, 200), rng.integers(0, hw0, 200), rng.integers(0, nd, 200)):
        fo, fn = c * hw0 + s, s * 512 + c
        sc, sh = fold(p["lin.b"], "bn0", fo)
        assert gw["lin"][0][fn, k] == _f2bf(f32(p["lin.w"][fo, k]) * sc)
        assert gw["lin"][1][fn] == sh
    S = ((0, 0), (1, 2)), ((0, 1), (2, 2))
    for layer, bn, co_n, ci_n in (("c1", "bn1", 256, 512), ("c2", "bn2", 128, 256)):
        w = p[layer + ".w"]
        for ph, co, ci, ty, tx in zip(rng.integers(0, 4, 300), rng.integers(0, co_n, 300), rng.integers(0, ci_n, 300),
                                      rng.integers(0, 2, 300), rng.integers(0, 2, 300)):
            a, b = ph >> 1, ph & 1
            total = 0.0
            for ky in range(S[a][ty][0], S[a][ty][1] + 1):
                for kx in range(S[b][tx][0], S[b][tx][1] + 1):
                    total += float(w[co, ci, ky, kx])
            sc, sh = fold(p[layer + ".b"], bn, co)
            assert gw[layer][0][a, b, co, ci, ty, tx] == _f2bf(f32(total * float(sc))), (layer, ph, co, ci, ty, tx)
            assert gw[layer][1][co] == sh
    for t in range(9):
        for co in range(C):
            for ci in range(0, 128, 7):
                assert gw["taps"][0][t * C + co, ci] == _f2bf(p["c3.w"][co, ci, t // 3, t % 3])
                assert gw["w3"][t * C + co, ci] == p["c3.w"][co, ci, t // 3, t % 3]


def test_R_weight_rounding_matches_load_R(pkg):
    """Loop-by-loop restatement of load_R_impl: conv1 f2bf(w * scale), convs f2bf(float(double(w) * scale)), Linear1
    wm[o][s*128 + c] = f2bf((0.75f * l1w[o][c*HWq + s]) * scale[o]), Linear2 f2bf(l2w) with shift l2b."""
    C, H, W, nd = 3, 32, 16, 6
    p = pkg.weights.unpack(pkg.weights.init_R(C, H, W, nd, seed=5, stress=True), pkg.weights.r_layout(C, H, W, nd))
    rw = tl.r_weights(p, C, H, W, nd)
    f32 = np.float32

    def fold(bias, bn, i):
        s = f32(p[bn + ".g"][i]) / f32(np.sqrt(f32(p[bn + ".v"][i] + f32(1e-5))))
        return s, f32(p[bn + ".b"][i] + f32(f32(bias[i]) - f32(p[bn + ".m"][i])) * s)

    rng = np.random.default_rng(6)
    for i, ci_n, co_n in ((1, C, 64), (2, 64, 64), (4, 64, 128), (6, 128, 128)):
        w = p[f"c{i}.w"]
        for co, ci, t in zip(rng.integers(0, co_n, 200), rng.integers(0, ci_n, 200), rng.integers(0, 9, 200)):
            sc, sh = fold(p[f"c{i}.b"], f"bn{i}", co)
            want = _f2bf(f32(w[co, ci, t // 3, t % 3]) * sc) if i == 1 else _f2bf(f32(float(w[co, ci, t // 3, t % 3]) * float(sc)))
            assert rw[f"c{i}"][0][co, ci, t // 3, t % 3] == want, (i, co, ci, t)
            assert rw[f"c{i}"][1][co] == sh
            if i == 1:
                assert rw["c1_simt"][0][co, ci, t // 3, t % 3] == w[co, ci, t // 3, t % 3] and rw["c1_simt"][1][co] == sc
    hwq = (H // 4) * (W // 4)
    for o, c, s in zip(rng.integers(0, 512, 300), rng.integers(0, 128, 300), rng.integers(0, hwq, 300)):
        sc, sh = fold(p["l1.b"], "bn7", o)
        assert rw["l1"][0][o, s * 128 + c] == _f2bf(f32(f32(0.75) * p["l1.w"][o, c * hwq + s]) * sc), (o, c, s)
        assert rw["l1"][1][o] == sh
    for k in range(nd):
        for c in range(0, 512, 11):
            assert rw["out"][0][k, c] == _f2bf(p["l2.w"][k, c])
        assert rw["out"][1][k] == p["l2.b"][k]

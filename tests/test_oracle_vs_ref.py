"""Pin the oracle restatement to the reference's OWN code: the reference's headers, compiled verbatim against the
Eigen / iod stand-ins in oracle/ref_shim, were run over the inputs below and their outputs stored in
tests/golden/reference_oracle_vs_ref.npz (tests/golden/make_reference_vectors.py); the oracle must reproduce them."""
import os

import numpy as np
import pytest

from tests import oracle as orc
from tests import reference_vectors as rv
from tests import scenes
from tests.oracle_ops import oracle_grad_pyramid, oracle_lk, oracle_lucas_kanade, oracle_pyramid

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def o(built):
    return orc.load()


@pytest.fixture(scope="module")
def G():
    return rv.load("oracle_vs_ref")


def rng(s):
    return np.random.default_rng(s)


# ---- inputs (shared with tests/golden/make_reference_vectors.py)
BORDER_PIXELS = ("u8", "vuchar3", "i32", "vint2")
PYRAMID_CASES = [(kind, pix, shape) for shape in [(101, 77), (100, 80)] for kind, pix in [(0, "u8"), (1, "vint2"), (2, "vfloat2")]]
LK_CASES = [(5, 2), (7, 2), (11, 2), (7, 1), (7, 3), (11, 3)]
SDOF_CASES = [((121, 161), 9, 3, 0, 2, 5), ((145, 209), 7, 4, 0, 2, 5), ((129, 97), 9, 3, 1, 3, 3), ((121, 161), 9, 2, 0, 0, 5)]
FAST9_MODES, FAST9_MASKS = (0, 1, 2), (None, 0xFF, 0x01, 0x10)


def add_inputs():
    b, c = rng(1).integers(-2 ** 30, 2 ** 30, (2, 37, 53), dtype=np.int32)
    return orc.HostImage(37, 53, "i32", aligned=16, data=b), orc.HostImage(37, 53, "i32", aligned=16, data=c)


def border_input(pix):
    dt, ch = orc.PIXEL_TYPES[pix]
    d = rng(2).integers(0, 200, (9, 14) + ((ch,) if ch > 1 else ())).astype(dt)
    return orc.HostImage(9, 14, pix, border=3, data=d)


def box_inputs():
    s = rng(3).integers(-1000, 1000, (41, 67), dtype=np.int32)
    u = rng(4).integers(0, 256, (45, 71, 3), dtype=np.uint8)
    return (orc.HostImage(41, 67, "i32", border=2, data=s, fill_border="mirror"),
            orc.HostImage(45, 71, "vuchar3", border=2, data=u, fill_border="mirror"))


def interp_input():
    a = rng(5).integers(0, 256, (33, 47), dtype=np.uint8)
    return orc.HostImage(33, 47, "u8", border=2, data=a, fill_border="mirror"), rng(6).uniform(0, 30, (200, 2)).astype(np.float32)


def pyramid_even_interior(x, shape, lvl):
    """even parent size: the last row/col of a level (and what mirrors / blurs it) is garbage in the reference
    (pyramid.hh:179-181); odd parent sizes and level 0 compare whole"""
    if shape[0] % 2 == 1 or lvl == 0:
        return x
    m = 3 + 4 * lvl
    return x[3:-m - 3, 3:-m - 3]


def fast9_cases():
    cases = [(scenes.rectangles_scene(131, 160, seed=seed), th) for seed, th in [(8, 10), (9, 20), (10, 40)]]
    # dense random patterns: pixels drawn from 3 levels exercise a large share of the 2^16 ring patterns
    cases.append((rng(11).choice(np.array([20, 100, 180], np.uint8), (96, 128)), 30))
    cases.append((rng(12).integers(0, 256, (64, 96), dtype=np.uint8), 15))
    return cases


def fast9_mask(img, maskval):
    if maskval is None:
        return None
    nr, nc = img.shape
    m = np.zeros(img.shape, np.uint8)
    m[5:nr - 9, 7:nc - 11] = maskval
    return orc.HostImage(nr, nc, "u8", aligned=32, data=m)


def lk_prediction(pred, n):
    return None if not pred else np.tile(np.array([[2.0, -2.0]], np.float32), (n, 1))


def sdof_inputs(shape, o):
    f1, f2, _ = scenes.lk_pair(shape[0], shape[1], 4, seed=21, shift=(3.0, -2.0), margin=10)
    k = np.zeros((f1.size, 2), np.int32)
    h = orc.HostImage(shape[0], shape[1], "u8", border=3, data=f1, fill_border="mirror")
    n = o.vo_fast9_u8(h.ptr(), 8, None, 2, 6, 0, k.ctypes.data, None, len(k))  # blockwise FAST keypoints, as video_extruder feeds it
    return f1, f2, np.ascontiguousarray(k[:n])


def rgb_input(pix, b):
    ch = 3 if pix == "vuchar3" else 4
    data = rng(77).integers(0, 256, (45, 67, ch), dtype=np.uint8)
    data[0, :, :3] = 255
    data[1, :, :3] = 0
    return orc.HostImage(45, 67, pix, border=b, aligned=32, data=data, fill_border="mirror" if b else None), data


def gray_kat():
    return (np.arange(100 * 100) % 256).astype(np.uint8).reshape(100, 100)


# ---- tests
def test_add_borders_box(G, o):
    hb, hc = add_inputs()
    a2 = orc.HostImage(37, 53, "i32", aligned=16)
    o.vo_pw_add_i32(a2.ptr(), hb.ptr(), hc.ptr())
    assert rv.digest(a2.get()) == G["add"]
    for pix in BORDER_PIXELS:
        h2 = border_input(pix)
        o.vo_fill_border_mirror(h2.ptr())
        assert rv.digest(h2.get(True)) == G["mirror_" + pix], pix
        if pix != "vint2":
            o.vo_fill_border_closest(h2.ptr())
            assert rv.digest(h2.get(True)) == G["closest_" + pix], pix
    hs, hu = box_inputs()
    d2 = orc.HostImage(41, 67, "i32")
    o.vo_box5x5_i32(hs.ptr(), d2.ptr())
    assert rv.digest(d2.get()) == G["box_i32"]
    d2 = orc.HostImage(45, 71, "vuchar3")
    o.vo_box5x5_u8(hu.ptr(), d2.ptr(), 3)
    assert rv.digest(d2.get()) == G["box_u8c3"]


def test_interp_scharr_lowpass(G, o):
    h, pts = interp_input()
    assert rv.digest(np.array([o.vo_interp_u8(h.ptr(), pr, pc) for (pr, pc) in pts], np.int64)) == G["interp"]
    for gpix in ("vint2", "vfloat2"):
        g2 = orc.HostImage(33, 47, gpix)
        o.vo_scharr_u8(h.ptr(), g2.ptr(), 1 if gpix == "vfloat2" else 0)
        assert rv.digest(g2.get().view(np.int32)) == G["scharr_" + gpix], gpix
    l2 = orc.HostImage(33, 47, "u8")
    o.vo_lowpass(h.ptr(), l2.ptr(), 0)
    assert rv.digest(l2.get()) == G["lowpass"]


@pytest.mark.parametrize("kind,pix", [(0, "u8"), (1, "vint2"), (2, "vfloat2")])
@pytest.mark.parametrize("shape", [(101, 77), (100, 80)])
def test_pyramids(G, o, kind, pix, shape):
    a = scenes.rectangles_scene(shape[0], shape[1], seed=7)
    mine = oracle_pyramid(a, 3, "u8", 3, o)
    if kind:
        mine = oracle_grad_pyramid(mine, pix, 3, o)
    for lvl in range(3):
        y = mine[lvl].get(True)
        if pix != "u8":
            y = y.view(np.int32)
        assert rv.digest(pyramid_even_interior(y, shape, lvl)) == G["pyramid_%d_%dx%d_L%d" % (kind, shape[0], shape[1], lvl)], "level %d" % lvl


@pytest.mark.parametrize("tree", ["scalar-tree", "avx2-tree"])
def test_fast9_reference_ring(G, o, tree):
    """The pruning tree of fast.hpp:253-508 (scalar fallback and the AVX2 build) == the oracle's 9-arc
    test on the ring as implemented; mask, threshold, maxima modes and scores included."""
    i = j = 0
    for img, th in fast9_cases():
        nr, nc = img.shape
        h = orc.HostImage(nr, nc, "u8", border=3, aligned=32, data=img, fill_border="mirror")
        for mode in FAST9_MODES:
            for maskval in FAST9_MASKS:
                hm = fast9_mask(img, maskval)
                k2, s2 = np.zeros((img.size, 2), np.int32), np.zeros(img.size, np.int32)
                n2 = o.vo_fast9_u8(h.ptr(), th, hm.ptr() if hm else None, mode, 10, 0, k2.ctypes.data, s2.ctypes.data, img.size)
                if mode == 2 and tree == "scalar-tree":  # serial build: the reference's own output order == the oracle's
                    assert rv.digest(np.array([n2]), k2[:n2]) == G["fast9_native"][j], (th, maskval)
                    j += 1
                if mode == 2:  # the oracle emits blockwise keypoints in cell order (the reference's serial order); the wrapper sorts by pixel
                    order = np.lexsort((k2[:n2, 1], k2[:n2, 0]))
                    k2[:n2], s2[:n2] = k2[:n2][order], s2[:n2][order]
                assert rv.digest(np.array([n2]), k2[:n2], s2[:n2]) == G["fast9_" + tree][i], (th, mode, maskval)
                i += 1
    assert i == len(G["fast9_" + tree]) and j == (len(G["fast9_native"]) if tree == "scalar-tree" else 0)


def test_fast9_true_ring_and_score(G, o):
    img = scenes.rectangles_scene(90, 120, seed=13)
    h = orc.HostImage(90, 120, "u8", border=3, data=img, fill_border="mirror")
    k = np.zeros((img.size, 2), np.int32)
    n = o.vo_fast9_u8(h.ptr(), 20, None, 0, 10, 1, k.ctypes.data, None, img.size)
    mine = k[:n][np.lexsort((k[:n, 1], k[:n, 0]))]  # raster order
    assert n > 20 and rv.digest(mine) == G["true_ring_kps"]
    assert rv.digest(np.array([o.vo_fast9_score(h.ptr(), 20, int(r_), int(c_)) for (r_, c_) in mine], np.int32)) == G["true_ring_scores"]


@pytest.mark.parametrize("winsize,nscales", LK_CASES)
def test_lucas_kanade_bit_exact(G, o, winsize, nscales):
    """lucas_kanade() of the reference vs the oracle: bit-identical flows and distances.  With 3 levels the
    reference's 4x overshoot at level 2 (blurred level-0 gradient, lucas_kanade.hpp:156-157) throws a few
    tracks against the image edge where its un-checked bilinear taps read outside the allocated border
    (undefined values; the oracle clamps): those (< 2 % of the points) are allowed to differ.  The reference's tracks are
    stored as a 16-bit digest each."""
    f1, f2, pts = scenes.lk_pair(301, 401, 400, seed=14, margin=40)
    for pred in (0, 1):
        rflow, rdist = oracle_lucas_kanade(f1, f2, pts, niterations=21, winsize=winsize, nscales=nscales, prediction=lk_prediction(pred, len(pts)), lib=o)
        bad = rv.point_digests(rflow, rdist) != G["lk_%d_%d_%d" % (winsize, nscales, pred)]
        if nscales <= 2:
            assert not bad.any(), bad.sum()
        else:
            assert bad.mean() < 0.02, bad.sum()


def test_reference_pyrlk_kat_through_real_headers(G, o):
    # tests/pyrlk.cc:14-50 executed by the reference's own lucas_kanade(), and the oracle on the same call
    d = np.load(os.path.join(ROOT, "tests", "golden", "pyrlk_scene.npz"))
    flow = G["pyrlk_kat_flow"]
    assert np.linalg.norm(flow[0] - np.array([2.0, 2.0])) < 0.05, flow
    mine, _ = oracle_lucas_kanade(d["i1"], d["i2"], np.array([[50, 50]], np.float32), niterations=50, winsize=5, nscales=2, min_ev=0.001, delta=0.01, lib=o)
    assert np.array_equal(flow.view(np.int32), mine.view(np.int32)), (flow, mine)


@pytest.mark.parametrize("winsize", [5, 7])
def test_lk_square_win_matcher(G, o, winsize):
    """lk_match_point_square_win<WS> (lk.hh:42-175) inside the pyrlk_match loop, float gradient pyramid."""
    f1, f2, pts = scenes.lk_pair(141, 181, 120, seed=15, margin=30)
    prev, nxt = oracle_pyramid(f1, 2, "u8", 4, o), oracle_pyramid(f2, 2, "u8", 4, o)
    grad = oracle_grad_pyramid(prev, "vfloat2", 4, o)
    flow, dist = G["lksq_%d_flow" % winsize], G["lksq_%d_dist" % winsize]
    P = orc.VoLkParams(nlevels=2, min_scale=0, winsize=winsize, max_iter=21, grad_is_float=1, err_mode=1, gate_on_max_err=1, min_ev=0.01, delta=0.01,
                       max_err=0.6, factor=2.0, pred_div=1.0)
    rflow, rdist = oracle_lk(prev, nxt, grad, P, pts, lib=o)
    assert np.array_equal(dist >= 3e38, rdist >= 3e38)
    assert np.allclose(flow, rflow, rtol=1e-5, atol=1e-5), np.abs(flow - rflow).max()
    ok = rdist < 3e38
    assert np.allclose(dist[ok], rdist[ok], rtol=1e-4)


@pytest.mark.parametrize("shape,ws,nscales,min_scale,prop,patch", SDOF_CASES)
def test_semi_dense_flow_serial_semantics(G, o, shape, ws, nscales, min_scale, prop, patch):
    """semi_dense_optical_flow (semi_dense_optical_flow.hpp:46-214 + gradient_descent.hh) executed by the reference's
    own headers, serial build, vs the oracle restatement: positions, distances and the set of reported keypoints.
    Sizes of the form 2^k m + 1 keep every pyramid level odd, so the reference never reads its uninitialised
    low-pass border (pyramid.hh:179-181)."""
    f1, f2, kps = sdof_inputs(shape, o)
    n = len(kps)
    assert n > 100
    h1, h2 = orc.HostImage(shape[0], shape[1], "u8", data=f1), orc.HostImage(shape[0], shape[1], "u8", data=f2)
    pos, dist, valid = np.zeros((n, 2), np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
    o.vo_semi_dense_flow(h1.ptr(), h2.ptr(), kps.ctypes.data, n, ws, nscales, min_scale, prop, patch, pos.ctypes.data, dist.ctypes.data, valid.ctypes.data)
    key = "sdof_%d" % SDOF_CASES.index((shape, ws, nscales, min_scale, prop, patch))
    assert rv.digest(valid) == G[key + "_valid"] and valid.sum() > 50
    assert rv.digest(pos) == G[key + "_pos"]
    assert rv.digest(dist) == G[key + "_dist"]
    flow = (pos - kps)[valid > 0]
    assert np.median(np.abs(flow - np.array([3, -2])).max(axis=1)) <= 1  # the synthetic motion is (3,-2) +- 0.5 px


def _moving_frames(nr, nc, nframes, seed=31):
    """a textured scene translating by (2,-1) px per frame (+ a little per-frame noise)"""
    base = scenes.rectangles_scene(nr + 64, nc + 64, seed=seed, noise=2)
    rngf = np.random.default_rng(seed)
    out = []
    for f in range(nframes):
        a = base[32 - 2 * f:32 - 2 * f + nr, 32 + f:32 + f + nc].astype(np.int32) + rngf.integers(-1, 2, (nr, nc))
        out.append(np.clip(a, 0, 255).astype(np.uint8))
    return out


def test_video_extruder_orchestration(G, o):
    """video_extruder_update (video_extruder.hpp:24-135) run by the reference's own headers over 7 frames (the -DNDEBUG
    build, one thread) vs the Python orchestration of vpp_b200.video_extruder on the oracle backend: identical keypoints,
    ages and trajectories."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("video_extruder", os.path.join(ROOT, "vpp_b200", "video_extruder.py"))
    ve = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ve)
    from tests.oracle_video import OracleOps

    nr, nc, nf = 161, 241, 7
    frames = _moving_frames(nr, nc, nf)
    ctx = ve.video_extruder_init(nr, nc)
    ops = OracleOps(o)
    for f in range(1, nf):
        ve.video_extruder_update(ctx, frames[f - 1], frames[f], ops, detector_th=6, keypoint_spacing=10, detector_period=3,
                                 max_trajectory_length=5, nscales=3, winsize=9, propagation=2)
    mine = ve.state_table(ctx)
    assert len(mine) > 20 and rv.digest(mine) == G["video_extruder"]
    assert (mine[:, 2] > 1).sum() > 5  # some keypoints really were tracked across frames


@pytest.mark.parametrize("pix", ["vuchar3", "vuchar4"])
def test_rgb_to_graylevel(G, o, pix):
    """rgb_to_graylevel<unsigned char> of the reference (colorspace_conversions.hh:22-47) vs the oracle: domain and border,
    every channel sum 0..765 occurs; + the reference's own KAT (tests/colorspace_conversions.cc:8-23): gray(i,i,i) == i."""
    for b in (0, 3):
        src, data = rgb_input(pix, b)
        g2 = orc.HostImage(45, 67, "u8", border=b, aligned=32)
        o.vo_rgb_to_graylevel(src.ptr(), g2.ptr())
        assert rv.digest(g2.get(True)) == G["gray_%s_b%d" % (pix, b)]
        assert np.array_equal(g2.get(), (data[..., :3].astype(np.int32).sum(axis=2) // 3).astype(np.uint8))
    if pix == "vuchar3":
        kat = gray_kat()
        src = orc.HostImage(100, 100, "vuchar3", data=np.repeat(kat[..., None], 3, axis=2))
        g = orc.HostImage(100, 100, "u8")
        o.vo_rgb_to_graylevel(src.ptr(), g.ptr())
        assert G["gray_v1_kat"] == rv.digest(kat) and np.array_equal(g.get(), kat)

"""SURVEY 8(f) N4 on the CPU: the oracle restatements of lbp_transform, local_maxima_filter, fast_detector9_blockwise_rank and the
oriented LK matcher against the reference's own test vector (tests/lbp.cc) and against what the reference's headers (lbp_transform.hh,
fast.hpp:555-575, lk.hh:180-317) computed on the same inputs, stored in tests/golden/reference_n4.npz by
tests/golden/make_reference_vectors.py (blockwise_rank is not instantiable in the reference - see the oracle)."""
import numpy as np
import pytest

from tests import oracle as orc
from tests import reference_vectors as rv
from tests import scenes
from tests.oracle_ops import oracle_grad_pyramid, oracle_pyramid

# stored random examples of the property pins below (drawn as in tests/test_oracle_vs_ref_property.py)
SPACES = {"lbp": dict(nr=(1, 30), nc=(1, 70), levels=(1, 255), aligned=[1, 4, 16, 128], seed=(0, 2 ** 16)),
          "lmf": dict(nr=(1, 24), nc=(1, 40), levels=(1, 40), pix=["u8", "i32"], signed=[False, True], seed=(0, 2 ** 16))}
EXAMPLES = {"lbp": 300, "lmf": 300}
LBP_SHAPES = [(3, 3), (37, 53), (64, 128), (5, 301)]
LMF_SHAPES = [(9, 14), (40, 67), (64, 96)]
ORIENTED_CASES = [(5, 10, 1.0), (7, 21, 0.5), (9, 15, 100.0), (11, 4, 2.0)]


@pytest.fixture(scope="module")
def o(built):
    return orc.load()


@pytest.fixture(scope="module")
def G():
    return rv.load("n4")


def test_lbp_known_answer(o):
    """tests/lbp.cc:9-38: the 3x3 image of the reference's test, lbp(1,1) == 0b10101110"""
    v = np.array([[0, 2, 2], [2, 1, 0], [2, 0, 2]], np.uint8)
    h = orc.HostImage(3, 3, "u8", border=1, data=v)
    out = orc.HostImage(3, 3, "u8")
    o.vo_lbp_u8(h.ptr(), out.ptr())
    assert out.get()[1, 1] == 0b10101110


def lbp_input(shape):
    img = np.random.default_rng(shape[1]).integers(0, 6, shape, dtype=np.uint8) * 40
    return orc.HostImage(shape[0], shape[1], "u8", border=1, data=img, fill_border="mirror")


@pytest.mark.parametrize("shape", LBP_SHAPES)
def test_lbp_equals_reference(G, o, shape):
    h = lbp_input(shape)
    b = orc.HostImage(shape[0], shape[1], "u8")
    o.vo_lbp_u8(h.ptr(), b.ptr())
    assert rv.digest(b.get()) == G["lbp_%dx%d" % shape] and len(np.unique(b.get())) > 3


def lmf_scenes(shape, pix, seed):
    """images that exercise the in-place dependence: plateaus, ramps (every pixel's left / upper neighbour is larger and gets zeroed first),
    sparse score-like images and dense noise"""
    r = np.random.default_rng(seed)
    nr, nc = shape
    hi = 250 if pix == "u8" else 100000
    out = [r.integers(0, hi, shape), r.integers(0, 4, shape), np.where(r.random(shape) < 0.05, r.integers(1, hi, shape), 0)]
    rr, cc = np.meshgrid(np.arange(nr), np.arange(nc), indexing="ij")
    out.append((hi - 1 - (rr + cc) % hi))             # decreasing along rows and columns: long chains of dependent decisions
    out.append(((rr * 3 + cc * 2) % 7) * (hi // 8))    # periodic ramps
    out.append(np.full(shape, 9))
    return [a.astype(np.uint8 if pix == "u8" else np.int32) for a in out]


@pytest.mark.parametrize("pix", ["u8", "i32"])
@pytest.mark.parametrize("shape", LMF_SHAPES)
def test_local_maxima_filter_serial_equals_reference(G, o, shape, pix):
    for i, img in enumerate(lmf_scenes(shape, pix, 3)):
        b = orc.HostImage(shape[0], shape[1], pix, border=1, data=img, fill_border="value")
        o.vo_local_maxima_filter(b.ptr())
        assert rv.digest(b.get(True)) == G["lmf_%s_%dx%d_%d" % ((pix,) + shape + (i,))], (i, pix)
        assert (b.get() != img).any() or i == 2


def oriented_case(nr, nc, n, seed, ws):
    f1, f2, pts = scenes.lk_pair(nr, nc, n, seed=seed, shift=(1.3, -0.8), margin=ws + 6)
    r = np.random.default_rng(seed)
    ang1, ang2 = r.uniform(0, 2 * np.pi, len(pts)), r.uniform(0, 2 * np.pi, len(pts))
    ang2[::2] = ang1[::2]  # half of the points search along the template's own direction
    d1 = np.stack([np.cos(ang1), np.sin(ang1)], axis=1).astype(np.float32)
    d2 = np.stack([np.cos(ang2), np.sin(ang2)], axis=1).astype(np.float32)
    d1[::5], d2[::5] = (0.0, 1.0), (0.0, 1.0)  # the axis-aligned window
    pred = r.uniform(-1.5, 1.5, (len(pts), 2)).astype(np.float32)
    pts = pts.copy()
    pts[:4] = [[1.5, 2.5], [nr - 2.0, nc - 3.0], [0.0, nc / 2], [nr / 2, 1.0]]  # windows that leave the domain
    return f1, f2, np.ascontiguousarray(pts, np.float32), pred, d1, d2


def oriented_inputs(ws, o):
    """frames (borders mirror-filled), float Scharr gradient of the first, keypoints, predictions and window directions"""
    nr, nc = 151, 203
    f1, f2, pts, pred, d1, d2 = oriented_case(nr, nc, 300, ws, ws)
    A = orc.HostImage(nr, nc, "u8", border=3, data=f1, fill_border="mirror")
    B = orc.HostImage(nr, nc, "u8", border=3, data=f2, fill_border="mirror")
    return A, B, oracle_grad_pyramid([A], "vfloat2", 3, o)[0], pts, pred, d1, d2


@pytest.mark.parametrize("ws,max_iter,max_step", ORIENTED_CASES)
def test_oriented_lk_equals_reference(G, o, ws, max_iter, max_step):
    A, B, Gr, pts, pred, d1, d2 = oriented_inputs(ws, o)
    n = len(pts)
    fb, eb = np.zeros((n, 2), np.float32), np.zeros(n, np.float32)
    o.vo_lk_match_oriented_u8(A.ptr(), B.ptr(), Gr.ptr(), 1, ws, 1e-3, max_iter, 0.01, max_step, pts.ctypes.data, pred.ctypes.data, d1.ctypes.data,
                              d2.ctypes.data, n, fb.ctypes.data, eb.ctypes.data)
    # points whose rotated windows leave the domain use uninitialised as[] / gs[] in the reference (zero here): the first four are not stored
    assert rv.digest(fb[4:], eb[4:]) == G["oriented_%d" % ws]
    ok = eb < 1e30
    assert ok.sum() > n // 2 and (np.abs(fb[ok] - np.array([1.3, -0.8])).max(axis=1) < 1.0).mean() > 0.5


def test_blockwise_rank_properties(o):
    """not instantiable in the reference: the restatement is checked against its own definition - every record is a strict 3x3 maximum of the
    raw score image inside its block, ranks are 0..k-1 in decreasing score order, and with max_points == 1 the rule keeps the LAST of
    the increasing maxima of the raster scan (a candidate replaces a smaller slot)"""
    img = scenes.rectangles_scene(120, 161, seed=3)
    h = orc.HostImage(120, 161, "u8", border=3, data=img, fill_border="mirror")
    cap = img.size
    for bs, mp in ((10, 3), (16, 1), (7, 16)):
        k3, sc = np.zeros((cap, 3), np.int32), np.zeros(cap, np.int32)
        n = o.vo_fast9_blockwise_rank(h.ptr(), 15, None, bs, mp, 0, k3.ctypes.data, sc.ctypes.data, cap)
        assert n > 20
        k3, sc = k3[:n], sc[:n]
        S = np.zeros((122, 163), np.int64)
        ka = np.zeros((cap, 2), np.int32)
        na = o.vo_fast9_u8(h.ptr(), 15, None, 0, bs, 0, ka.ctypes.data, None, cap)
        for (r, c) in ka[:na]:
            S[r + 1, c + 1] = o.vo_fast9_score(h.ptr(), 15, int(r), int(c))
        for (r, c, k), s in zip(k3, sc):
            win = S[r:r + 3, c:c + 3].copy()
            assert s == win[1, 1] and s > 0
            win[1, 1] = -1
            assert s > win.max() and 0 <= k < mp
        blocks = (k3[:, 0] // bs) * 1000 + k3[:, 1] // bs
        assert (np.diff(blocks) >= 0).all()  # blocks in raster order
        for b in np.unique(blocks):
            m = blocks == b
            assert list(k3[m, 2]) == list(range(m.sum())) or mp > 1 and (np.diff(k3[m, 2]) > 0).all()
            assert (np.diff(sc[m]) <= 0).all()


# ---- property pins over stored random examples (SPACES above): random geometries and value ranges
def lbp_any_input(nr, nc, levels, aligned, seed):
    img = np.random.default_rng(seed).integers(0, levels + 1, (nr, nc)).astype(np.uint8)
    return orc.HostImage(nr, nc, "u8", border=1, aligned=aligned, data=img, fill_border="value", border_value=seed % 256)


def lmf_any_input(nr, nc, levels, pix, signed, seed):
    lo = -levels if (signed and pix == "i32") else 0
    img = np.random.default_rng(seed).integers(lo, levels + 1, (nr, nc)).astype(np.uint8 if pix == "u8" else np.int32)
    return orc.HostImage(nr, nc, pix, border=1, data=img, fill_border="value", border_value=seed % 5)


def test_lbp_any_geometry(G, o):
    for i, p in rv.cases(SPACES, EXAMPLES, "lbp"):
        h = lbp_any_input(**p)
        b = orc.HostImage(p["nr"], p["nc"], "u8", aligned=p["aligned"])
        o.vo_lbp_u8(h.ptr(), b.ptr())
        assert rv.digest(b.get()) == G["lbp_digest"][i], p


def test_local_maxima_filter_any_image(G, o):
    """few grey levels = many ties and plateaus: the strict comparisons and the in-place order decide everything"""
    for i, p in rv.cases(SPACES, EXAMPLES, "lmf"):
        b = lmf_any_input(**p)
        o.vo_local_maxima_filter(b.ptr())
        assert rv.digest(b.get(True)) == G["lmf_digest"][i], p

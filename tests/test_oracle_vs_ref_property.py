"""Pinning of the oracle against the reference's own headers over random geometries: ragged sizes, borders, alignments,
thresholds, masks.  tests/golden/make_reference_vectors.py ran the reference on the examples drawn from SPACES and stored its outputs
in tests/golden/reference_property.npz; here the oracle must reproduce them.  CPU only."""
import numpy as np
import pytest

from tests import oracle as orc
from tests import reference_vectors as rv

# parameter spaces and counts of the stored examples (see tests/reference_vectors.cases)
SPACES = {
    "border": dict(nr=(1, 40), nc=(1, 60), border=(0, 6), aligned=[1, 4, 16, 32, 128], pix=["u8", "vuchar3", "i32", "vint2"], seed=(0, 2 ** 16)),
    "box": dict(nr=(1, 40), nc=(1, 50), aligned=[1, 16, 32, 128], seed=(0, 2 ** 16), kind=["i32", "vuchar3"]),
    "scharr": dict(nr=(3, 45), nc=(3, 60), seed=(0, 2 ** 16), as_float=[False, True]),
    "pyramid": dict(kr=(4, 12), kc=(4, 12), seed=(0, 2 ** 16), kind=[0, 1, 2], border=(2, 4)),
    "fast9": dict(nr=(8, 48), nc=(8, 70), th=(0, 80), seed=(0, 2 ** 16), mode=[0, 1, 2], bs=(2, 12), maskval=[None, 0xFF, 0x01, 0x10, 0x11, 0x80],
                  levels=[2, 3, 256]),
    "lk": dict(seed=(0, 2 ** 16), winsize=[5, 7, 9, 11, 15], nscales=[1, 2], niter=(1, 30), sr=(-3.0, 3.0), sc=(-3.0, 3.0), min_ev=[0.0001, 0.01, 1.0],
               delta=[0.01, 0.1, 0.5]),
    "sdof": dict(seed=(0, 2 ** 16), ws=[5, 7, 9, 11], nscales=(1, 3), min_scale=(0, 1), prop=(0, 3), patch=[3, 5], nk=(1, 400)),
}
EXAMPLES = {"border": 1500, "box": 1500, "scharr": 1500, "pyramid": 1500, "fast9": 1500, "lk": 300, "sdof": 150}


@pytest.fixture(scope="module")
def o(built):
    return orc.load()


@pytest.fixture(scope="module")
def G():
    return rv.load("property")


def _img(seed, nr, nc, pix, border, aligned, lo=0, hi=256):
    dt, ch = orc.PIXEL_TYPES[pix]
    d = np.random.default_rng(seed).integers(lo, hi, (nr, nc) + ((ch,) if ch > 1 else ())).astype(dt)
    return orc.HostImage(nr, nc, pix, border=border, aligned=aligned, data=d), d


def box_input(o, nr, nc, aligned, seed, kind):
    b = min(2 + seed % 3, max(nr, 2), max(nc, 2))
    if nr < 2 or nc < 2:
        b = 2  # mirror needs border <= size; tiny images are filled by value instead
    hs, _ = _img(seed, nr, nc, kind, b, aligned, -500 if kind == "i32" else 0, 1000 if kind == "i32" else 256)
    if b <= nr and b <= nc:
        o.vo_fill_border_mirror(hs.ptr())
    else:
        v = np.zeros(4, np.int32)
        o.vo_fill_border_value(hs.ptr(), v.ctypes.data)
    return hs


def scharr_input(o, nr, nc, seed):
    h, _ = _img(seed, nr, nc, "u8", 2, 16)
    o.vo_fill_border_mirror(h.ptr())
    return h


def fast9_input(nr, nc, seed, maskval, levels):
    r = np.random.default_rng(seed)
    img = (r.integers(0, levels, (nr, nc)) * (255 // max(levels - 1, 1))).astype(np.uint8)
    h = orc.HostImage(nr, nc, "u8", border=3, aligned=32, data=img, fill_border="mirror")
    hm = None
    if maskval is not None:
        m = (r.integers(0, 2, (nr, nc)) * maskval).astype(np.uint8)
        hm = orc.HostImage(nr, nc, "u8", aligned=32, data=m)
    return h, hm, img.size


def lk_input(seed, sr, sc):
    from tests import scenes

    nr, nc = 101 + 2 * (seed % 20), 121 + 2 * (seed % 17)
    f1, f2, pts = scenes.lk_pair(nr, nc, 60, seed=seed, shift=(sr, sc), margin=30)
    return f1, f2, pts


def lk_small(flow):
    """tracks that stayed small: the synthetic motion is <= 3 px"""
    return np.abs(np.nan_to_num(flow, nan=1e9, posinf=1e9, neginf=1e9)).max(axis=1) <= 8


def sdof_input(seed, nk):
    from tests import scenes

    nr, nc = 97, 129  # 2^5 * m + 1: every level odd
    r = np.random.default_rng(seed)
    f1, f2, _ = scenes.lk_pair(nr, nc, 4, seed=seed, shift=(float(r.integers(-3, 4)), float(r.integers(-3, 4))), margin=10)
    kps = np.stack([r.integers(0, nr, nk), r.integers(0, nc, nk)], axis=1).astype(np.int32)
    return orc.HostImage(nr, nc, "u8", data=f1), orc.HostImage(nr, nc, "u8", data=f2), kps


def sdof_outputs(pos, dist, valid):
    ok = valid > 0
    return rv.digest(valid, pos[ok], dist[ok])


def test_border_fills_any_geometry(G, o):
    for i, p in rv.cases(SPACES, EXAMPLES, "border"):
        border = min(p["border"], p["nr"], p["nc"])
        h2, _ = _img(p["seed"], p["nr"], p["nc"], p["pix"], border, p["aligned"])
        o.vo_fill_border_mirror(h2.ptr())
        outs = [h2.get(True)]
        if p["pix"] != "vint2":
            o.vo_fill_border_closest(h2.ptr())
            outs.append(h2.get(True))
        assert rv.digest(*outs) == G["border_digest"][i], p


def test_box_any_geometry(G, o):
    for i, p in rv.cases(SPACES, EXAMPLES, "box"):
        nr, nc, kind = p["nr"], p["nc"], p["kind"]
        hs = box_input(o, nr, nc, p["aligned"], p["seed"], kind)
        d2 = orc.HostImage(nr, nc, kind, aligned=p["aligned"])
        if kind == "i32":
            o.vo_box5x5_i32(hs.ptr(), d2.ptr())
        else:
            o.vo_box5x5_u8(hs.ptr(), d2.ptr(), 3)
        assert rv.digest(d2.get()) == G["box_digest"][i], p


def test_scharr_and_lowpass_any_geometry(G, o):
    for i, p in rv.cases(SPACES, EXAMPLES, "scharr"):
        nr, nc = p["nr"], p["nc"]
        h = scharr_input(o, nr, nc, p["seed"])
        g2 = orc.HostImage(nr, nc, "vfloat2" if p["as_float"] else "vint2")
        o.vo_scharr_u8(h.ptr(), g2.ptr(), int(p["as_float"]))
        l2 = orc.HostImage(nr, nc, "u8")
        o.vo_lowpass(h.ptr(), l2.ptr(), 0)
        assert rv.digest(g2.get().view(np.int32), l2.get()) == G["scharr_digest"][i], p


def test_pyramids_odd_safe_sizes(G, o):
    """sizes 4k+1 keep all three levels free of the reference's uninitialised low-pass border"""
    from tests.oracle_ops import oracle_grad_pyramid, oracle_pyramid

    for i, p in rv.cases(SPACES, EXAMPLES, "pyramid"):
        nr, nc = 4 * p["kr"] + 1, 4 * p["kc"] + 1
        a = np.random.default_rng(p["seed"]).integers(0, 256, (nr, nc), dtype=np.uint8)
        pix = ["u8", "vint2", "vfloat2"][p["kind"]]
        mine = oracle_pyramid(a, 3, "u8", p["border"], o)
        if p["kind"]:
            mine = oracle_grad_pyramid(mine, pix, p["border"], o)
        levels = [l.get(True) if pix == "u8" else l.get(True).view(np.int32) for l in mine]
        assert rv.digest(*levels) == G["pyramid_digest"][i], p


def test_fast9_any_geometry(G, o):
    for i, p in rv.cases(SPACES, EXAMPLES, "fast9"):
        h, hm, size = fast9_input(p["nr"], p["nc"], p["seed"], p["maskval"], p["levels"])
        k2, s2 = np.zeros((size, 2), np.int32), np.zeros(size, np.int32)
        n2 = o.vo_fast9_u8(h.ptr(), p["th"], hm.ptr() if hm else None, p["mode"], p["bs"], 0, k2.ctypes.data, s2.ctypes.data, size)
        if p["mode"] == 2:
            order = np.lexsort((k2[:n2, 1], k2[:n2, 0]))
            k2[:n2], s2[:n2] = k2[:n2][order], s2[:n2][order]
        assert rv.digest(np.array([n2]), k2[:n2], s2[:n2]) == G["fast9_digest"][i], p


def test_lucas_kanade_any_parameters(G, o):
    """reference lucas_kanade() vs the oracle, bit for bit, over random scenes, window sizes, iteration caps and thresholds.
    winsize 3 is left out: lucas_kanade.hpp:149 gives the pyramids a border of winsize/2 = 1, and the 5-tap low-pass of
    pyramid.hh:179-181 then reads 2 pixels out — past the border, undefined values (the CUDA path refuses it: VPPB_E_BORDER).
    The reference's tracks are stored as a 16-bit digest each (a changed track goes unnoticed with probability 2^-16)."""
    from tests.oracle_ops import oracle_lucas_kanade

    for i, p in rv.cases(SPACES, EXAMPLES, "lk"):
        f1, f2, pts = lk_input(p["seed"], p["sr"], p["sc"])
        nr, nc = f1.shape
        rflow, rdist = oracle_lucas_kanade(f1, f2, pts, niterations=p["niter"], winsize=p["winsize"], nscales=p["nscales"], min_ev=p["min_ev"],
                                           delta=p["delta"], lib=o)
        # A track that diverges wanders to the image edge, where the reference's un-checked bilinear taps read past the
        # allocated border (undefined values; the oracle clamps) - it may even come back.  Such tracks are recognisable by
        # their size: the synthetic motion is <= 3 px.  Every track that stayed small on both sides and ends well inside the
        # image must match bit for bit; the others must be rare.
        end = pts + rflow
        m = p["winsize"] // 2 + 2
        inside = (end[:, 0] >= m) & (end[:, 0] <= nr - 1 - m) & (end[:, 1] >= m) & (end[:, 1] <= nc - 1 - m) & np.isfinite(end).all(axis=1)
        small = G["lk_small"][i] & lk_small(rflow)
        same = rv.point_digests(rflow, rdist) == G["lk_points"][i]
        sane = inside & small
        assert sane.mean() > 0.5, p
        assert same[sane].all(), p
        assert (~same).mean() < 0.1, p


def test_semi_dense_flow_any_parameters(G, o):
    """random keypoint sets (duplicates and several keypoints per cell included, any order): the first-claim,
    Gauss-Seidel propagation and reporting rules of the reference's serial build, bit for bit"""
    for i, p in rv.cases(SPACES, EXAMPLES, "sdof"):
        nscales, nk = p["nscales"], p["nk"]
        min_scale = min(p["min_scale"], nscales - 1)
        h1, h2, kps = sdof_input(p["seed"], nk)
        pos, dist, valid = np.zeros((nk, 2), np.int32), np.zeros(nk, np.int32), np.zeros(nk, np.uint8)
        o.vo_semi_dense_flow(h1.ptr(), h2.ptr(), kps.ctypes.data, nk, p["ws"], nscales, min_scale, p["prop"], p["patch"], pos.ctypes.data, dist.ctypes.data,
                             valid.ctypes.data)
        assert sdof_outputs(pos, dist, valid) == G["sdof_digest"][i], p

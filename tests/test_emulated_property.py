"""Property-based sweeps (hypothesis, derandomized) of the CUDA kernels on the CPU emulator against the oracle: geometries
and parameters nobody would write down by hand - strip widths around the 992-byte tile, row counts around the 8 / 16
row tiles, one-pixel images, thresholds, masks, window sizes, keypoints on the frame edge."""
import ctypes as C
import gc
import os
import sys

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from tests import oracle as orc
from tests import scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCALE = float(os.environ.get("VPPB_PROPERTY_SCALE", "1"))  # > 1 for a longer sweep (the numbers below x SCALE examples)
SET = dict(deadline=None, derandomize=True, suppress_health_check=[HealthCheck.function_scoped_fixture, HealthCheck.too_slow])


@pytest.fixture(scope="module")
def vpp(built):
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu

    emu = C.CDLL(build_emu.build())
    import vpp_b200
    from vpp_b200 import capi, ops

    for name, (res, args) in capi.PROTOTYPES.items():
        fn = getattr(emu, name)
        fn.restype, fn.argtypes = res, args
    ops._FAST_CACHE.clear()  # cached FAST workspaces are freed by the library that allocated them (tests/test_emulated_parity.py)
    mp = pytest.MonkeyPatch()
    mp.setattr(capi, "lib", emu)
    mp.setattr(ops, "lib", emu)
    yield vpp_b200
    ops._FAST_CACHE.clear()
    gc.collect()
    mp.undo()


def _box_oracle(data, pix):
    ch = 3 if pix == "vuchar3" else 1
    hs = orc.HostImage(data.shape[0], data.shape[1], pix, border=2, data=data, fill_border="mirror")
    hd = orc.HostImage(data.shape[0], data.shape[1], pix)
    orc.load().vo_box5x5_u8(hs.ptr(), hd.ptr(), ch)
    return hd.get()


# widths whose byte rows end just before / on / after a 992-byte strip and a 16-byte store group
WIDTHS = st.one_of(st.integers(1, 40), st.sampled_from([330, 331, 332, 661, 662, 663, 992, 993, 1000]), st.integers(320, 345))


@settings(max_examples=int(150 * SCALE), **SET)
@given(nr=st.one_of(st.integers(1, 40), st.sampled_from([47, 48, 49, 63, 64, 65])), nc=WIDTHS, pix=st.sampled_from(["vuchar3", "u8"]), seed=st.integers(0, 1000),
       extreme=st.sampled_from([None, 0, 255]))
def test_box_single(vpp, nr, nc, pix, seed, extreme):
    if nr < 2 or nc < 2:
        nr, nc = max(nr, 2), max(nc, 2)  # the mirror border of 2 needs 2 pixels
    ch = 3 if pix == "vuchar3" else 1
    shape = (nr, nc) + ((ch,) if ch > 1 else ())
    data = np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8) if extreme is None else np.full(shape, extreme, np.uint8)
    S = vpp.Image2d.from_host(data, pix, border=2)
    vpp.fill_border_mirror(S)
    D = vpp.Image2d(nr, nc, pix)
    vpp.box5x5(S, D)
    assert np.array_equal(D.download(), _box_oracle(data, pix)), (nr, nc, pix)


@settings(max_examples=int(40 * SCALE), **SET)
@given(nr=st.integers(2, 70), nc=st.one_of(st.integers(2, 60), st.integers(325, 340)), n=st.integers(2, 35), pix=st.sampled_from(["vuchar3", "u8"]), seed=st.integers(0, 1000))
def test_box_batch(vpp, nr, nc, n, pix, seed):
    ch = 3 if pix == "vuchar3" else 1
    r = np.random.default_rng(seed)
    uniq = [r.integers(0, 256, (nr, nc) + ((ch,) if ch > 1 else ()), dtype=np.uint8) for _ in range(min(n, 3))]
    exp = [_box_oracle(u, pix) for u in uniq]
    srcs, dsts = [], []
    for i in range(n):
        S = vpp.Image2d.from_host(uniq[i % len(uniq)], pix, border=2)
        vpp.fill_border_mirror(S)
        srcs.append(S)
        dsts.append(vpp.Image2d(nr, nc, pix))
    vpp.box5x5_batch(srcs, dsts)
    for i in range(n):
        assert np.array_equal(dsts[i].download(), exp[i % len(uniq)]), (i, nr, nc, n)


@settings(max_examples=int(150 * SCALE), **SET)
@given(nr=st.integers(1, 60), nc=st.integers(1, 90), th=st.integers(0, 120), seed=st.integers(0, 1000), mode=st.sampled_from([0, 1, 2]), bs=st.integers(1, 15),
       ring=st.sampled_from([0, 1]), maskval=st.sampled_from([None, 0xFF, 0x01, 0x10, 0x11]), levels=st.sampled_from([2, 4, 256]))
def test_fast9(vpp, nr, nc, th, seed, mode, bs, ring, maskval, levels):
    nr, nc = max(nr, 3), max(nc, 3)  # the mirror border of 3
    r = np.random.default_rng(seed)
    img = (r.integers(0, levels, (nr, nc)) * (255 // max(levels - 1, 1))).astype(np.uint8)
    mask = None if maskval is None else (r.integers(0, 2, (nr, nc)) * maskval).astype(np.uint8)
    o = orc.load()
    h = orc.HostImage(nr, nc, "u8", border=3, data=img, fill_border="mirror")
    hm = orc.HostImage(nr, nc, "u8", data=mask) if mask is not None else None
    k, sc = np.zeros((img.size, 2), np.int32), np.zeros(img.size, np.int32)
    n = o.vo_fast9_u8(h.ptr(), th, hm.ptr() if hm else None, mode, bs, ring, k.ctypes.data, sc.ctypes.data, img.size)
    G = vpp.Image2d.from_host(img, "u8", border=3)
    vpp.fill_border_mirror(G)
    got_sc = []
    got = vpp.fast9(G, th, mask=vpp.Image2d.from_host(mask, "u8") if mask is not None else None, local_maxima=mode == 1, blockwise=mode == 2, block_size=bs,
                    ring="true" if ring else "reference", scores=got_sc)
    assert len(got) == n and np.array_equal(got, k[:n]), (nr, nc, th, mode, bs, ring, maskval)
    assert np.array_equal(np.asarray(got_sc, np.int32), sc[:n])


@settings(max_examples=int(5 * SCALE), **SET)
@given(seed=st.integers(0, 1000), winsize=st.sampled_from([5, 7, 9, 11, 13, 15]), nscales=st.sampled_from([1, 2, 3]), niter=st.integers(1, 25), edge=st.booleans(),
       sr=st.floats(-3, 3), sc=st.floats(-3, 3))
def test_lucas_kanade(vpp, seed, winsize, nscales, niter, edge, sr, sc):
    """the LK kernels (4 keypoints per warp up to WS 11, one warp per keypoint above) replay the oracle's float evaluation
    order: flows and distances are compared bit for bit, failure codes included; keypoints on the frame edge included"""
    from tests.oracle_ops import oracle_lucas_kanade

    nr, nc = 97 + 2 * (seed % 9), 129 + 2 * (seed % 7)
    f1, f2, pts = scenes.lk_pair(nr, nc, 40, seed=seed, shift=(sr, sc), margin=4 if edge else 25)
    if edge:
        pts = np.concatenate([pts, np.array([[0, 0], [nr - 1, nc - 1], [0, nc // 2], [nr // 2, 0]], np.float32)])
    flow, dist = vpp.lucas_kanade(vpp.Image2d.from_host(f1, "u8"), vpp.Image2d.from_host(f2, "u8"), pts, niterations=niter, winsize=winsize, nscales=nscales)
    rflow, rdist = oracle_lucas_kanade(f1, f2, pts, niterations=niter, winsize=winsize, nscales=nscales)
    assert np.array_equal(flow.view(np.int32), rflow.view(np.int32)), np.nanmax(np.abs(flow - rflow))
    assert np.array_equal(dist.view(np.int32), rdist.view(np.int32))


@settings(max_examples=int(25 * SCALE), **SET)
@given(seed=st.integers(0, 1000), ws=st.sampled_from([5, 7, 9, 11]), nscales=st.integers(1, 3), min_scale=st.integers(0, 1), prop=st.integers(0, 3), patch=st.sampled_from([3, 5, 7]),
       nk=st.integers(1, 300))
def test_semi_dense_flow(vpp, seed, ws, nscales, min_scale, prop, patch, nk):
    min_scale = min(min_scale, nscales - 1)
    nr, nc = 97, 129
    r = np.random.default_rng(seed)
    f1, f2, _ = scenes.lk_pair(nr, nc, 4, seed=seed, shift=(float(r.integers(-3, 4)), float(r.integers(-3, 4))), margin=10)
    kps = np.stack([r.integers(0, nr, nk), r.integers(0, nc, nk)], axis=1).astype(np.int32)
    pos, dist, valid = vpp.semi_dense_optical_flow(kps, vpp.Image2d.from_host(f1, "u8"), vpp.Image2d.from_host(f2, "u8"), winsize=ws, nscales=nscales,
                                                   min_scale=min_scale, propagation=prop, patchsize=patch)
    h1, h2 = orc.HostImage(nr, nc, "u8", data=f1), orc.HostImage(nr, nc, "u8", data=f2)
    rpos, rdist, rvalid = np.zeros((nk, 2), np.int32), np.zeros(nk, np.int32), np.zeros(nk, np.uint8)
    orc.load().vo_semi_dense_flow(h1.ptr(), h2.ptr(), kps.ctypes.data, nk, ws, nscales, min_scale, prop, patch, rpos.ctypes.data, rdist.ctypes.data, rvalid.ctypes.data)
    assert np.array_equal(valid, rvalid.astype(bool))
    ok = rvalid > 0
    assert np.array_equal(pos[ok], rpos[ok]) and np.array_equal(dist[ok], rdist[ok])


# ---- SURVEY 8(f) N4 stencils -----------------------------------------------------------------------------------------------------
@settings(max_examples=int(80 * SCALE), **SET)
@given(nr=st.integers(1, 23), nc=st.one_of(st.integers(1, 50), st.sampled_from([15, 16, 17, 31, 32, 33, 47, 48, 49, 64, 65])), levels=st.integers(1, 255),
       aligned=st.sampled_from([4, 16, 128]), seed=st.integers(0, 1000))
def test_lbp_transform(vpp, nr, nc, levels, aligned, seed):
    """widths around the 16-pixel vectors of the kernel (full vectors, the ragged right edge, images narrower than one vector), row counts
    around its 4-row strips, 16-byte aligned and unaligned rows"""
    img = np.random.default_rng(seed).integers(0, levels + 1, (nr, nc)).astype(np.uint8)
    A = vpp.Image2d.from_host(img, "u8", border=1, aligned=aligned)
    vpp.fill_border_with_value(A, seed % 256)
    B = vpp.lbp_transform(A, vpp.Image2d(nr, nc, "u8", aligned=aligned))
    h = orc.HostImage(nr, nc, "u8", border=1, aligned=aligned, data=img, fill_border="value", border_value=seed % 256)
    r = orc.HostImage(nr, nc, "u8", aligned=aligned)
    orc.load().vo_lbp_u8(h.ptr(), r.ptr())
    assert np.array_equal(B.download(), r.get())


@settings(max_examples=int(60 * SCALE), **SET)
@given(nr=st.integers(1, 20), nc=st.one_of(st.integers(1, 40), st.sampled_from([15, 16, 17, 32, 33])), levels=st.integers(1, 30), pix=st.sampled_from(["u8", "i32"]),
       signed=st.booleans(), seed=st.integers(0, 1000))
def test_local_maxima_filter(vpp, nr, nc, levels, pix, signed, seed):
    """few grey levels (ties, plateaus, chains of dependent decisions across the 16-pixel runs of the kernel), signed values, any border value:
    the relaxation passes must land on the serial raster-order result"""
    lo = -levels if (signed and pix == "i32") else 0
    img = np.random.default_rng(seed).integers(lo, levels + 1, (nr, nc)).astype(np.uint8 if pix == "u8" else np.int32)
    bv = seed % 5
    A = vpp.Image2d.from_host(img, pix, border=1)
    vpp.fill_border_with_value(A, bv)
    vpp.local_maxima_filter(A)
    h = orc.HostImage(nr, nc, pix, border=1, data=img, fill_border="value", border_value=bv)
    orc.load().vo_local_maxima_filter(h.ptr())
    assert np.array_equal(A.download(with_border=True), h.get(True))


@settings(max_examples=int(25 * SCALE), **SET)
@given(nr=st.integers(8, 60), nc=st.integers(8, 90), th=st.integers(2, 60), bs=st.integers(1, 24), mp=st.integers(1, 16), ring=st.sampled_from(["reference", "true"]),
       masked=st.booleans(), seed=st.integers(0, 1000))
def test_fast9_blockwise_rank(vpp, nr, nc, th, bs, mp, ring, masked, seed):
    """fast_detector9_blockwise_rank: any block size (1 pixel to larger than the image), table sizes 1 .. 16, both rings, masks"""
    img = scenes.rectangles_scene(nr, nc, seed=seed, nrect=max(4, nr * nc // 150))
    G = vpp.Image2d.from_host(img, "u8", border=3)
    vpp.fill_border_mirror(G)
    h = orc.HostImage(nr, nc, "u8", border=3, data=img, fill_border="mirror")
    M = hm = None
    if masked:
        m = np.random.default_rng(seed).choice(np.array([0, 0x01, 0x10, 0xFF], np.uint8), (nr, nc))
        M, hm = vpp.Image2d.from_host(m, "u8"), orc.HostImage(nr, nc, "u8", data=m)
    sc = []
    got = vpp.fast9_blockwise_rank(G, th, block_size=bs, max_points_per_block=mp, mask=M, scores=sc, ring=ring)
    cap = nr * nc * 2
    k3, s = np.zeros((cap, 3), np.int32), np.zeros(cap, np.int32)
    n = orc.load().vo_fast9_blockwise_rank(h.ptr(), th, hm.ptr() if hm else None, bs, mp, 0 if ring == "reference" else 1, k3.ctypes.data, s.ctypes.data, cap)
    assert n >= 0 and len(got) == n
    assert np.array_equal(got, k3[:n]) and np.array_equal(np.array(sc, np.int32).reshape(-1), s[:n])

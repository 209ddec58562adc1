"""Reference vectors for tests/test_oracle_vs_ref.py, tests/test_oracle_vs_ref_property.py and tests/test_n4_oracle.py: the
reference's own headers, compiled verbatim against the Eigen / iod stand-ins of oracle/ref_shim (oracle/_ref/libvppref.so: serial,
-O2, scalar FAST tree; libvppref_omp.so: the reference's benchmark flags, AVX2 FAST tree), run over the inputs those tests build.
Needs the reference tree and oracle/_ref (oracle/ref_shim/build_ref.sh); run from the repository root:
    python tests/golden/make_reference_vectors.py
Writes tests/golden/reference_{oracle_vs_ref,property,n4}.npz (read through tests/reference_vectors.py): digests of the outputs the
tests compare exactly, values where they allow a tolerance."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import oracle as orc  # noqa: E402
from tests import reference_vectors as rv  # noqa: E402
from tests import scenes  # noqa: E402
from tests import test_n4_oracle as N4  # noqa: E402
from tests import test_oracle_vs_ref as T  # noqa: E402
from tests import test_oracle_vs_ref_property as P  # noqa: E402
from tests.oracle_ops import oracle_grad_pyramid, oracle_pyramid  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "libvppref.so")
REF_OMP = os.path.join(ROOT, "oracle", "_ref", "libvppref_omp.so")
I = C.POINTER(orc.VoImg)


def load_ref(path):
    r = C.CDLL(path)
    r.vppref_pw_add_i32.argtypes = [I, I, I]
    r.vppref_fill_border_mirror.argtypes = [I]
    r.vppref_fill_border_closest.argtypes = [I]
    r.vppref_box5x5_i32.argtypes = [I, I]
    r.vppref_box5x5_u8c3.argtypes = [I, I]
    r.vppref_scharr_u8.argtypes = [I, I, C.c_int]
    r.vppref_rgb_to_graylevel.argtypes = [I, I]
    r.vppref_rgb_to_graylevel_v1.argtypes = [I, I]
    r.vppref_lowpass_u8.argtypes = [I, I]
    r.vppref_pyramid.argtypes = [I, C.c_int, I, C.c_int]
    r.vppref_fast9_u8.argtypes = [I, C.c_int, I, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    r.vppref_fast9_blockwise_native_order.argtypes = [I, C.c_int, I, C.c_int, C.c_void_p, C.c_int]
    r.vppref_fast9_score.argtypes = [I, C.c_int, C.c_int, C.c_int]
    r.vppref_is_fast9_keypoint.argtypes = [I, C.c_int, C.c_int, C.c_int]
    r.vppref_interp_u8.argtypes = [I, C.c_float, C.c_float]
    r.vppref_lucas_kanade.argtypes = [I, I, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
    r.vppref_video_extruder.argtypes = [I, C.c_int] + [C.c_int] * 7 + [C.c_void_p, C.c_int]
    r.vppref_semi_dense_flow.argtypes = [I, I, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    r.vppref_pyrlk_levels.argtypes = [I, I, I, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float,
                                      C.c_void_p, C.c_void_p]
    r.vppref_lbp_u8.argtypes = [I, I]
    r.vppref_local_maxima_filter.argtypes = [I]
    r.vppref_lk_match_oriented.argtypes = [I, I, I, C.c_int, C.c_float, C.c_int, C.c_float, C.c_float] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_void_p]
    return r


def oracle_vs_ref(ref, ref_omp, o):
    G = {}
    hb, hc = T.add_inputs()
    a1 = orc.HostImage(37, 53, "i32", aligned=16)
    ref.vppref_pw_add_i32(a1.ptr(), hb.ptr(), hc.ptr())
    G["add"] = rv.digest(a1.get())
    for pix in T.BORDER_PIXELS:
        h1 = T.border_input(pix)
        ref.vppref_fill_border_mirror(h1.ptr())
        G["mirror_" + pix] = rv.digest(h1.get(True))
        if pix != "vint2":
            ref.vppref_fill_border_closest(h1.ptr())
            G["closest_" + pix] = rv.digest(h1.get(True))
    hs, hu = T.box_inputs()
    d1 = orc.HostImage(41, 67, "i32")
    ref.vppref_box5x5_i32(hs.ptr(), d1.ptr())
    G["box_i32"] = rv.digest(d1.get())
    d1 = orc.HostImage(45, 71, "vuchar3")
    ref.vppref_box5x5_u8c3(hu.ptr(), d1.ptr())
    G["box_u8c3"] = rv.digest(d1.get())

    h, pts = T.interp_input()
    G["interp"] = rv.digest(np.array([ref.vppref_interp_u8(h.ptr(), pr, pc) for (pr, pc) in pts], np.int64))
    for gpix in ("vint2", "vfloat2"):
        g1 = orc.HostImage(33, 47, gpix)
        ref.vppref_scharr_u8(h.ptr(), g1.ptr(), 1 if gpix == "vfloat2" else 0)
        G["scharr_" + gpix] = rv.digest(g1.get().view(np.int32))
    l1 = orc.HostImage(33, 47, "u8")
    ref.vppref_lowpass_u8(h.ptr(), l1.ptr())
    G["lowpass"] = rv.digest(l1.get())

    for kind, pix, shape in T.PYRAMID_CASES:
        a = scenes.rectangles_scene(shape[0], shape[1], seed=7)
        src = orc.HostImage(shape[0], shape[1], "u8", data=a)
        mine = oracle_pyramid(a, 3, "u8", 3, o)  # level geometry only
        theirs = [orc.HostImage(l.nrows, l.ncols, pix, border=3) for l in mine]
        ref.vppref_pyramid(src.ptr(), 3, orc.desc_array(theirs), kind)
        for lvl in range(3):
            x = theirs[lvl].get(True)
            G["pyramid_%d_%dx%d_L%d" % (kind, shape[0], shape[1], lvl)] = rv.digest(T.pyramid_even_interior(x if pix == "u8" else x.view(np.int32), shape, lvl))

    native = []
    for tree, r in (("scalar-tree", ref), ("avx2-tree", ref_omp)):
        res = []
        for img, th in T.fast9_cases():
            nr, nc = img.shape
            h = orc.HostImage(nr, nc, "u8", border=3, aligned=32, data=img, fill_border="mirror")
            for mode in T.FAST9_MODES:
                for maskval in T.FAST9_MASKS:
                    hm = T.fast9_mask(img, maskval)
                    k1, s1 = np.zeros((img.size, 2), np.int32), np.zeros(img.size, np.int32)
                    n1 = r.vppref_fast9_u8(h.ptr(), th, hm.ptr() if hm else None, mode, 10, k1.ctypes.data, s1.ctypes.data, img.size)
                    res.append(rv.digest(np.array([n1]), k1[:n1], s1[:n1]))
                    if mode == 2 and tree == "scalar-tree":
                        k3 = np.zeros((img.size, 2), np.int32)
                        n3 = r.vppref_fast9_blockwise_native_order(h.ptr(), th, hm.ptr() if hm else None, 10, k3.ctypes.data, img.size)
                        native.append(rv.digest(np.array([n3]), k3[:n3]))
        G["fast9_" + tree] = np.array(res, np.uint64)
    G["fast9_native"] = np.array(native, np.uint64)

    img = scenes.rectangles_scene(90, 120, seed=13)
    h = orc.HostImage(90, 120, "u8", border=3, data=img, fill_border="mirror")
    kps = np.array([(r_, c_) for r_ in range(90) for c_ in range(120) if ref.vppref_is_fast9_keypoint(h.ptr(), 20, r_, c_)], np.int32)
    G["true_ring_kps"] = rv.digest(kps)
    G["true_ring_scores"] = rv.digest(np.array([ref.vppref_fast9_score(h.ptr(), 20, int(r_), int(c_)) for (r_, c_) in kps], np.int32))

    f1, f2, pts = scenes.lk_pair(301, 401, 400, seed=14, margin=40)
    h1, h2 = orc.HostImage(301, 401, "u8", data=f1), orc.HostImage(301, 401, "u8", data=f2)
    n = len(pts)
    for winsize, nscales in T.LK_CASES:
        for pred in (0, 1):
            p_ = T.lk_prediction(pred, n)
            flow, dist = np.zeros((n, 2), np.float32), np.zeros(n, np.float32)
            ref.vppref_lucas_kanade(h1.ptr(), h2.ptr(), pts.ctypes.data, p_.ctypes.data if p_ is not None else None, n, 21, winsize, nscales,
                                    0.0001, 0.1, flow.ctypes.data, dist.ctypes.data)
            G["lk_%d_%d_%d" % (winsize, nscales, pred)] = rv.point_digests(flow, dist)

    d = np.load(os.path.join(ROOT, "tests", "golden", "pyrlk_scene.npz"))
    h1, h2 = orc.HostImage(100, 100, "u8", data=d["i1"]), orc.HostImage(100, 100, "u8", data=d["i2"])
    kp = np.array([[50, 50]], np.float32)
    flow, dist = np.zeros((1, 2), np.float32), np.zeros(1, np.float32)
    ref.vppref_lucas_kanade(h1.ptr(), h2.ptr(), kp.ctypes.data, None, 1, 50, 5, 2, 0.001, 0.01, flow.ctypes.data, dist.ctypes.data)
    G["pyrlk_kat_flow"] = flow

    f1, f2, pts = scenes.lk_pair(141, 181, 120, seed=15, margin=30)
    prev, nxt = oracle_pyramid(f1, 2, "u8", 4, o), oracle_pyramid(f2, 2, "u8", 4, o)
    grad = oracle_grad_pyramid(prev, "vfloat2", 4, o)
    n = len(pts)
    for winsize in (5, 7):
        flow, dist = np.zeros((n, 2), np.float32), np.zeros(n, np.float32)
        ref.vppref_pyrlk_levels(orc.desc_array(prev), orc.desc_array(nxt), orc.desc_array(grad), 2, 0, winsize, pts.ctypes.data, n, 0.01, 0.6, 21.0, 0.01,
                                flow.ctypes.data, dist.ctypes.data)
        G["lksq_%d_flow" % winsize], G["lksq_%d_dist" % winsize] = flow, dist

    for i, (shape, ws, nscales, min_scale, prop, patch) in enumerate(T.SDOF_CASES):
        f1, f2, kps = T.sdof_inputs(shape, o)
        n = len(kps)
        h1, h2 = orc.HostImage(shape[0], shape[1], "u8", data=f1), orc.HostImage(shape[0], shape[1], "u8", data=f2)
        pos, dist, valid = np.zeros((n, 2), np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
        ref.vppref_semi_dense_flow(h1.ptr(), h2.ptr(), kps.ctypes.data, n, ws, nscales, min_scale, prop, patch, pos.ctypes.data, dist.ctypes.data, valid.ctypes.data)
        G["sdof_%d_pos" % i], G["sdof_%d_dist" % i], G["sdof_%d_valid" % i] = rv.digest(pos), rv.digest(dist), rv.digest(valid)

    # video_extruder_update with the -DNDEBUG build, one thread (serial semantics): with asserts on, keypoint_container.hpp:82 aborts
    # as soon as a dead keypoint is revived by move() - which the reference's own update loop does (video_extruder.hpp:48-51)
    ref_omp.vppref_set_num_threads(1)
    nr, nc, nf = 161, 241, 7
    hosts = [orc.HostImage(nr, nc, "u8", border=10, aligned=32, data=f, fill_border="mirror") for f in T._moving_frames(nr, nc, nf)]
    out = np.zeros((nr * nc, 6), np.int32)
    n = ref_omp.vppref_video_extruder(orc.desc_array(hosts), nf, 6, 10, 3, 5, 3, 9, 2, out.ctypes.data, len(out))
    G["video_extruder"] = rv.digest(out[:n])

    for pix in ("vuchar3", "vuchar4"):
        for b in (0, 3):
            src, _ = T.rgb_input(pix, b)
            g1 = orc.HostImage(45, 67, "u8", border=b, aligned=32)
            ref.vppref_rgb_to_graylevel(src.ptr(), g1.ptr())
            G["gray_%s_b%d" % (pix, b)] = rv.digest(g1.get(True))
    kat = T.gray_kat()
    src = orc.HostImage(100, 100, "vuchar3", data=np.repeat(kat[..., None], 3, axis=2))
    g = orc.HostImage(100, 100, "u8")
    ref.vppref_rgb_to_graylevel_v1(src.ptr(), g.ptr())
    G["gray_v1_kat"] = rv.digest(g.get())
    return G


def prop_border(ref, o, p):
    border = min(p["border"], p["nr"], p["nc"])
    h1, _ = P._img(p["seed"], p["nr"], p["nc"], p["pix"], border, p["aligned"])
    ref.vppref_fill_border_mirror(h1.ptr())
    outs = [h1.get(True)]
    if p["pix"] != "vint2":
        ref.vppref_fill_border_closest(h1.ptr())
        outs.append(h1.get(True))
    return rv.digest(*outs)


def prop_box(ref, o, p):
    nr, nc, kind = p["nr"], p["nc"], p["kind"]
    hs = P.box_input(o, nr, nc, p["aligned"], p["seed"], kind)
    d1 = orc.HostImage(nr, nc, kind, aligned=p["aligned"])
    (ref.vppref_box5x5_i32 if kind == "i32" else ref.vppref_box5x5_u8c3)(hs.ptr(), d1.ptr())
    return rv.digest(d1.get())


def prop_scharr(ref, o, p):
    nr, nc = p["nr"], p["nc"]
    h = P.scharr_input(o, nr, nc, p["seed"])
    g1 = orc.HostImage(nr, nc, "vfloat2" if p["as_float"] else "vint2")
    ref.vppref_scharr_u8(h.ptr(), g1.ptr(), int(p["as_float"]))
    l1 = orc.HostImage(nr, nc, "u8")
    ref.vppref_lowpass_u8(h.ptr(), l1.ptr())
    return rv.digest(g1.get().view(np.int32), l1.get())


def prop_pyramid(ref, o, p):
    nr, nc = 4 * p["kr"] + 1, 4 * p["kc"] + 1
    a = np.random.default_rng(p["seed"]).integers(0, 256, (nr, nc), dtype=np.uint8)
    pix = ["u8", "vint2", "vfloat2"][p["kind"]]
    src = orc.HostImage(nr, nc, "u8", data=a)
    theirs = [orc.HostImage(l.nrows, l.ncols, pix, border=p["border"]) for l in oracle_pyramid(a, 3, "u8", p["border"], o)]
    ref.vppref_pyramid(src.ptr(), 3, orc.desc_array(theirs), p["kind"])
    return rv.digest(*[l.get(True) if pix == "u8" else l.get(True).view(np.int32) for l in theirs])


def prop_fast9(ref, o, p):
    h, hm, size = P.fast9_input(p["nr"], p["nc"], p["seed"], p["maskval"], p["levels"])
    k1, s1 = np.zeros((size, 2), np.int32), np.zeros(size, np.int32)
    n1 = ref.vppref_fast9_u8(h.ptr(), p["th"], hm.ptr() if hm else None, p["mode"], p["bs"], k1.ctypes.data, s1.ctypes.data, size)
    return rv.digest(np.array([n1]), k1[:n1], s1[:n1])


def prop_lk(ref, o, p):
    f1, f2, pts = P.lk_input(p["seed"], p["sr"], p["sc"])
    nr, nc = f1.shape
    h1, h2 = orc.HostImage(nr, nc, "u8", data=f1), orc.HostImage(nr, nc, "u8", data=f2)
    n = len(pts)
    flow, dist = np.zeros((n, 2), np.float32), np.zeros(n, np.float32)
    ref.vppref_lucas_kanade(h1.ptr(), h2.ptr(), pts.ctypes.data, None, n, p["niter"], p["winsize"], p["nscales"], p["min_ev"], p["delta"], flow.ctypes.data,
                            dist.ctypes.data)
    return rv.point_digests(flow, dist), P.lk_small(flow)


def prop_sdof(ref, o, p):
    nscales, nk = p["nscales"], p["nk"]
    h1, h2, kps = P.sdof_input(p["seed"], nk)
    pos, dist, valid = np.zeros((nk, 2), np.int32), np.zeros(nk, np.int32), np.zeros(nk, np.uint8)
    ref.vppref_semi_dense_flow(h1.ptr(), h2.ptr(), kps.ctypes.data, nk, p["ws"], nscales, min(p["min_scale"], nscales - 1), p["prop"], p["patch"],
                               pos.ctypes.data, dist.ctypes.data, valid.ctypes.data)
    return P.sdof_outputs(pos, dist, valid)


def prop_lbp(ref, o, p):
    h = N4.lbp_any_input(**p)
    a = orc.HostImage(p["nr"], p["nc"], "u8", aligned=p["aligned"])
    ref.vppref_lbp_u8(h.ptr(), a.ptr())
    return rv.digest(a.get())


def prop_lmf(ref, o, p):
    a = N4.lmf_any_input(**p)
    ref.vppref_local_maxima_filter(a.ptr())
    return rv.digest(a.get(True))


def properties(ref, o, spaces, examples, fns):
    G = {}
    for name in spaces:
        res = [fns[name](ref, o, p) for _, p in rv.cases(spaces, examples, name)]
        if name == "lk":
            G["lk_points"], G["lk_small"] = np.stack([r_[0] for r_ in res]), np.stack([r_[1] for r_ in res])
        else:
            G[name + "_digest"] = np.array(res, np.uint64)
    return G


def n4(ref, o):
    G = {}
    for shape in N4.LBP_SHAPES:
        a = orc.HostImage(shape[0], shape[1], "u8")
        ref.vppref_lbp_u8(N4.lbp_input(shape).ptr(), a.ptr())
        G["lbp_%dx%d" % shape] = rv.digest(a.get())
    for pix in ("u8", "i32"):
        for shape in N4.LMF_SHAPES:
            for i, img in enumerate(N4.lmf_scenes(shape, pix, 3)):
                a = orc.HostImage(shape[0], shape[1], pix, border=1, data=img, fill_border="value")
                ref.vppref_local_maxima_filter(a.ptr())
                G["lmf_%s_%dx%d_%d" % ((pix,) + shape + (i,))] = rv.digest(a.get(True))
    for ws, max_iter, max_step in N4.ORIENTED_CASES:
        A, B, Gr, pts, pred, d1, d2 = N4.oriented_inputs(ws, o)
        n = len(pts)
        fa, ea = np.zeros((n, 2), np.float32), np.zeros(n, np.float32)
        ref.vppref_lk_match_oriented(A.ptr(), B.ptr(), Gr.ptr(), ws, 1e-3, max_iter, 0.01, max_step, pts.ctypes.data, pred.ctypes.data, d1.ctypes.data,
                                     d2.ctypes.data, n, fa.ctypes.data, ea.ctypes.data)
        # the first four windows leave the domain: the reference reads uninitialised values there
        G["oriented_%d" % ws] = rv.digest(fa[4:], ea[4:])
    return G


if __name__ == "__main__":
    ref, ref_omp, o = load_ref(REF), load_ref(REF_OMP), orc.load()
    fns = dict(border=prop_border, box=prop_box, scharr=prop_scharr, pyramid=prop_pyramid, fast9=prop_fast9, lk=prop_lk, sdof=prop_sdof, lbp=prop_lbp, lmf=prop_lmf)
    out = {"oracle_vs_ref": oracle_vs_ref(ref, ref_omp, o), "property": properties(ref, o, P.SPACES, P.EXAMPLES, fns),
           "n4": {**n4(ref, o), **properties(ref, o, N4.SPACES, N4.EXAMPLES, fns)}}
    for name, G in out.items():
        path = os.path.join(ROOT, "tests", "golden", "reference_%s.npz" % name)
        np.savez_compressed(path, **G)
        print(path, os.path.getsize(path), "bytes")

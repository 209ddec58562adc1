"""Golden fixture for the C++ video_extruder test (tests/cpp/extruder_tests.cu): 9 frames of a translating scene in
which a flat occluder appears at frame 3 (corners under it fade) and a patch is mirrored from frame 5 (the flow goes
astray there), and the keypoint / trajectory tables that the REFERENCE's own video_extruder_update (compiled from
/root/reference through oracle/ref_shim, -DNDEBUG, one thread) leaves after 7 frames (detector_th 4) and after
9 frames (detector_th 5).  Run in the build container (needs /root/reference):
    python tests/golden/make_video_extruder_fixture.py
Writes video_extruder_frames_9x121x161.u8 (raw frames, row-major) and video_extruder_expected_{7f_th4,9f_th5}.i32
(rows of: row, col, age, trajectory start frame, trajectory length, trajectory alive)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import oracle as orc  # noqa: E402
from tests import scenes  # noqa: E402

NR, NC, NF = 121, 161, 9
CASES = {"7f_th4": (7, 4), "9f_th5": (9, 5)}
OTHER = dict(keypoint_spacing=10, detector_period=3, max_trajectory_length=5, nscales=3, winsize=9, propagation=2)


def eventful_frames(nr=NR, nc=NC, nf=NF, seed=77):
    base = scenes.rectangles_scene(nr + 96, nc + 96, seed=seed, noise=2)
    r = np.random.default_rng(seed)
    out = []
    for f in range(nf):
        a = base[48 - 3 * f:48 - 3 * f + nr, 48 + 2 * f:48 + 2 * f + nc].astype(np.int32) + r.integers(-1, 2, (nr, nc))
        a = np.clip(a, 0, 255).astype(np.uint8)
        if f >= 3:
            a[20:70, 30:110] = 128
        if f >= 5:
            a[80:, :60] = a[80:, :60][:, ::-1]
        out.append(a)
    return out


def reference_table(frames, nframes, detector_th):
    from tests.golden.make_reference_vectors import REF_OMP, load_ref

    ref = load_ref(REF_OMP)
    ref.vppref_set_num_threads(1)
    nr, nc = frames[0].shape
    hosts = [orc.HostImage(nr, nc, "u8", border=10, aligned=32, data=f, fill_border="mirror") for f in frames[:nframes]]
    out = np.zeros((nr * nc, 6), np.int32)
    n = ref.vppref_video_extruder(orc.desc_array(hosts), nframes, detector_th, OTHER["keypoint_spacing"], OTHER["detector_period"],
                                  OTHER["max_trajectory_length"], OTHER["nscales"], OTHER["winsize"], OTHER["propagation"], out.ctypes.data, len(out))
    return out[:n].copy()


if __name__ == "__main__":
    frames = eventful_frames()
    here = os.path.dirname(os.path.abspath(__file__))
    np.stack(frames).astype(np.uint8).tofile(os.path.join(here, "video_extruder_frames_%dx%dx%d.u8" % (NF, NR, NC)))
    for tag, (nf, th) in CASES.items():
        t = reference_table(frames, nf, th)
        t.tofile(os.path.join(here, "video_extruder_expected_%s.i32" % tag))
        print(tag, "keypoints", len(t), "tracked (age > 1)", int((t[:, 2] > 1).sum()), "dead", int((t[:, 2] == 0).sum()), "starts", np.unique(t[:, 3]).tolist())

#!/usr/bin/env python
"""A/B timing of the 5x5 box byte kernels (GPU box only): one child process per variant (the kernel choice is read from
the environment once per process), CUDA events on the launch stream, image sets larger than L2.
Usage: python tools/box_bench.py > gpurun_out/box_bench.json"""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = [
    ("default", {}),
    ("tile", {"VPPB_BOX_IMPL": "tile"}),
    ("stream_single", {"VPPB_BOX_SINGLE": "stream"}),
]


def child():
    import numpy as np
    import torch

    import vpp_b200 as vpp
    from vpp_b200 import capi

    capi.check(capi.lib.vppb_init(0))
    peak = 6564.5
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        peak = json.load(open(p))["hbm_gbs"]
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    rng = np.random.default_rng(0)
    out = {}

    def timed(fn, reps):
        fn(); fn(); fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / reps  # us per call of fn

    for (H, W, tag, pix, cs) in [(1080, 1920, "1080p", "vuchar3", 3), (2160, 3840, "4k", "vuchar3", 3), (4320, 7680, "8k", "vuchar3", 3),
                                 (2160, 3840, "4k_u8", "u8", 1)]:
        alg = 2.0 * cs * H * W
        n = max(2, int(np.ceil(1600e6 / alg)))
        n = min(n, 128)
        f = rng.integers(0, 256, (H, W, cs) if cs > 1 else (H, W), dtype=np.uint8)
        S = [vpp.Image2d.from_host(f, pix, border=2) for _ in range(n)]
        D = [vpp.Image2d(H, W, pix) for _ in range(n)]
        for s in S:
            vpp.fill_border_mirror(s)
        one = capi.lib.vppb_box5x5_u8c3 if cs == 3 else capi.lib.vppb_box5x5_u8
        bat = capi.lib.vppb_box5x5_u8c3_batch if cs == 3 else capi.lib.vppb_box5x5_u8_batch

        def per_frame():
            for i in range(n):
                capi.check(one(S[i].ptr(), D[i].ptr(), sp))

        us = timed(per_frame, 20) / n
        out["single_" + tag] = {"us_per_frame": round(us, 2), "frac": round(alg / (us * 1e-6) / 1e9 / peak, 3)}
        bi, bo = (capi.VppbImg * n)(*[x.desc for x in S]), (capi.VppbImg * n)(*[x.desc for x in D])
        us = timed(lambda: capi.check(bat(bi, bo, n, sp)), 20) / n
        out["batch%d_" % n + tag] = {"us_per_frame": round(us, 2), "frac": round(alg / (us * 1e-6) / 1e9 / peak, 3)}
        del S, D
    print(json.dumps(out))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "child":
        child()
        sys.exit(0)
    res = {}
    for name, env in VARIANTS:
        e = dict(os.environ)
        e.update(env)
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "child"], env=e, capture_output=True, text=True, timeout=300)
            res[name] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as ex:  # noqa: BLE001
            res[name] = {"error": repr(ex)}
        print(name, json.dumps(res[name]), file=sys.stderr)
    print(json.dumps(res, indent=1))

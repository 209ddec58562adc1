#!/usr/bin/env python
"""bench.py - the hot path of BASELINE.json on N B200s of one node, one JSON line on stdout.

Headline metric: Mpix/s of the 5x5 box filter on image2d<vuchar3> (BASELINE configs[1]).
  --gpus 1 : 1920x1080 vuchar3 frames.  128 frame pairs are resident (1.6 GB >> the 126 MB L2); a STEP filters
             PASSES x 128 frames (>= 5 ms of GPU work): one vppb_box5x5_u8c3_batch call per 128 frames = one launch of
             the per-warp streaming kernel (TMA ring per warp), the whole step replayed as a CUDA graph.
  --gpus N : 7680x4320 vuchar3 frames row-tiled over N ranks (one tile per GPU and frame).  A step filters PASSES x 32 frames
             with vppb_box5x5_u8c3_tiles: the kernel pulls the 2 halo rows above / below each tile straight from the
             neighbour GPU's memory (CUDA IPC mapping, bulk copies inside its own TMA pipeline) - compute and halo transfer
             are ONE kernel, there is no exchange step.  Same frames for every N > 1 ("strong"); the single-GPU figure of the
             same 8K workload is measured in the N = 1 run (extras.box5x5_vuchar3_8k_x32 = scaling_anchor_n1).
  value  : whole-job Mpix/s with inputs resident in HBM (CUDA events on the launch stream, max over ranks).
  e2e    : same metric through the C-ABI with HOST buffers (pinned): upload + mirror border fill + box5x5 + download inside
           the timed region, for every frame of the step.
  extras : (N = 1) pixel_wise add 4K, single-launch 4K box, 8K batch, frame ingest, FAST9 4K, pyrLK 1080p/10k, semi-dense flow -
           each with `parity` (checked against the oracle in this run) and a reference-kind CPU figure beside it.
--impl reference times the reference's own CPU implementation (oracle/_ref = the reference headers compiled with its
benchmark flags -O3 -march=native -fopenmp; the oracle port only if that library is missing) on the host cores.
--dump-outputs DIR writes what the timed step computed (see dump_outputs) so that two builds can be compared output for output;
the inputs are seeded, identical from run to run.
The bench runs from the tree build() left and writes nothing into it.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # no __pycache__ in the tree: it may be read-only
sys.path.insert(0, ROOT)

WORKLOADS = {"1080p": (1080, 1920), "4k": (2160, 3840), "8k": (4320, 7680)}
BOX_BYTES_PER_PX = 6.0  # algorithmic: 3 B read + 3 B written per vuchar3 pixel (SURVEY 8d)
BATCH_1GPU, BATCH_TILED = 128, 32  # resident frame pairs = frames per launch (1080p frames at N = 1, 8K row tiles at N > 1)
DUMP_BYTES = 48e6  # --dump-outputs budget over all ranks (at most 64 MB)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    """Threads the CPU arm may use: logical CPUs, clipped by affinity and by the cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def make_frames(h, w, nframes, seed=42):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(nframes)]


# ------------------------------------------------------------------------------------------ CPU arm
class CpuRef:
    """The reference's own code on the host cores: oracle/_ref/libvppref_omp.so (kind "reference": the reference headers compiled
    verbatim with its benchmark flags); the C port of the oracle (kind "port") only where that library is missing."""

    def __init__(self):
        from tests import oracle as orc

        self.orc = orc
        self.port = orc.load(omp=True)
        self.ref = None
        path = os.path.join(ROOT, "oracle", "_ref", "libvppref_omp.so")
        if os.path.exists(path):
            try:
                r = C.CDLL(path)
                I, P = C.POINTER(orc.VoImg), C.c_void_p
                r.vppref_box5x5_u8c3.argtypes = [I, I]
                r.vppref_pw_add_i32.argtypes = [I, I, I]
                r.vppref_fast9_u8.argtypes = [I, C.c_int, I, C.c_int, C.c_int, P, P, C.c_int]
                r.vppref_pyrlk_levels.argtypes = [I, I, I, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, P, P]
                r.vppref_semi_dense_flow.argtypes = [I, I, P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, P, P]
                r.vppref_num_threads.restype = C.c_int
                self.ref = r
            except Exception:
                self.ref = None
        self.threads = host_threads()
        self.set_threads(self.threads)

    def set_threads(self, n):
        self.port.vo_set_num_threads(n)
        if self.ref is not None:
            self.ref.vppref_set_num_threads(n)
        self.threads = n

    def pick_threads(self, fn):
        """All the host threads the reference can use: the full count and half of it (SMT), the faster is kept."""
        best, best_t, full = None, None, host_threads()
        for n in sorted({full, max(1, full // 2)}, reverse=True):
            self.set_threads(n)
            fn()
            times, t_end = [], time.perf_counter() + 0.6  # ~0.6 s per candidate, the fastest repetition counts (robust to a noisy start)
            while len(times) < 5 or time.perf_counter() < t_end:
                t0 = time.perf_counter()
                fn()
                times.append(time.perf_counter() - t0)
                if len(times) >= 400:
                    break
            dt = min(times)
            if best_t is None or dt < best_t:
                best, best_t = n, dt
        self.set_threads(best)
        return best

    @property
    def kind(self):
        return "reference" if self.ref is not None else "port"


def timed_cpu(fn, budget_s, max_reps=1000):
    fn()
    t0, reps = time.perf_counter(), 0
    while reps < 1 or (time.perf_counter() - t0 < budget_s and reps < max_reps):
        fn()
        reps += 1
    return (time.perf_counter() - t0) / reps


def cpu_box_bench(h, w, steps, warmup, budget_s):
    """Reference CPU path for the headline workload: image2d<vuchar3> 5x5 box (examples/box_filter.cc form), OpenMP over rows."""
    cpu = CpuRef()
    orc = cpu.orc
    fn = cpu.ref.vppref_box5x5_u8c3 if cpu.ref is not None else (lambda a, b: cpu.port.vo_box5x5_u8(a, b, 3))
    src = make_frames(h, w, 1)[0]
    hs = orc.HostImage(h, w, "vuchar3", border=2, aligned=32, data=src, fill_border="mirror")
    hd = orc.HostImage(h, w, "vuchar3", aligned=32)
    cores = cpu.pick_threads(lambda: fn(hs.ptr(), hd.ptr()))
    fn(hs.ptr(), hd.ptr())
    t0 = time.perf_counter()
    fn(hs.ptr(), hd.ptr())
    one = time.perf_counter() - t0
    per_step = max(1, min(4096, int(budget_s / max(one, 1e-4) / max(steps + warmup, 1))))  # ~budget_s seconds of CPU work in total
    for _ in range(warmup):
        for _ in range(per_step):
            fn(hs.ptr(), hd.ptr())
    t0 = time.perf_counter()
    for _ in range(steps):
        for _ in range(per_step):
            fn(hs.ptr(), hd.ptr())
    dt = time.perf_counter() - t0
    mpix = steps * per_step * h * w / 1e6 / dt
    return {"value": mpix, "unit": "Mpix/s", "cores": int(cores), "kind": cpu.kind,
            "sample": "%d frames of %dx%d vuchar3 per step x %d steps (%.1f s)" % (per_step, w, h, steps, dt)}, dt / steps * 1e3


def cpu_extras(budget_s=10.0):
    """The reference's own code (kind "reference") for the other rows of the path, bounded samples, all host threads."""
    from tests import scenes
    from tests.oracle_ops import oracle_grad_pyramid, oracle_pyramid

    cpu = CpuRef()
    orc, o, r = cpu.orc, cpu.port, cpu.ref
    out = {"cores": cpu.threads, "kind": cpu.kind}
    share = budget_s / 4.0
    # pixel_wise add, 4K int32 (benchmarks/image_add.cc)
    b = np.random.default_rng(1).integers(0, 2 ** 30, (2, 2160, 3840), dtype=np.int32)
    ha, hb, hc = (orc.HostImage(2160, 3840, "i32", aligned=32), orc.HostImage(2160, 3840, "i32", aligned=32, data=b[0]),
                  orc.HostImage(2160, 3840, "i32", aligned=32, data=b[1]))
    add = (lambda: r.vppref_pw_add_i32(ha.ptr(), hb.ptr(), hc.ptr())) if r is not None else (lambda: o.vo_pw_add_i32(ha.ptr(), hb.ptr(), hc.ptr()))
    s = timed_cpu(add, share)
    out["add_i32_4k"] = {"mpix_per_s": 2160 * 3840 / 1e6 / s, "kind": cpu.kind, "cores": cpu.threads}
    # FAST9 4K (fast.hpp:253-508, AVX2 pruning tree in the reference build)
    img = scenes.rectangles_scene(2160, 3840, seed=42)
    hg = orc.HostImage(2160, 3840, "u8", border=3, aligned=32, data=img, fill_border="mirror")
    cap = img.size // 4
    kps = np.zeros((cap, 2), dtype=np.int32)
    fast = (lambda: r.vppref_fast9_u8(hg.ptr(), 20, None, 0, 10, kps.ctypes.data, None, cap)) if r is not None else \
        (lambda: o.vo_fast9_u8(hg.ptr(), 20, None, 0, 10, 0, kps.ctypes.data, None, cap))
    s = timed_cpu(fast, share)
    out["fast9_4k"] = {"mpix_per_s": 2160 * 3840 / 1e6 / s, "ms": s * 1e3, "kind": cpu.kind, "cores": cpu.threads}
    # pyrLK 1080p, 3 levels, 10k keypoints, 7x7: the pyrlk_match loop (OpenMP over keypoints, pyrlk_match.hh:24) around lk_match_point_square_win<7>
    f1, f2, pts = scenes.lk_pair(1080, 1920, 10000, seed=5)
    prev, nxt = oracle_pyramid(f1, 3, "u8", 4, o), oracle_pyramid(f2, 3, "u8", 4, o)
    grad = oracle_grad_pyramid(prev, "vfloat2", 4, o)
    n = len(pts)
    flow, dist = np.zeros((n, 2), np.float32), np.zeros(n, np.float32)
    kp = np.ascontiguousarray(pts, dtype=np.float32)
    if r is not None:
        lk = lambda: r.vppref_pyrlk_levels(orc.desc_array(prev), orc.desc_array(nxt), orc.desc_array(grad), 3, 0, 7, kp.ctypes.data, n, 0.01, 0.6, 21.0, 0.01,
                                           flow.ctypes.data, dist.ctypes.data)
    else:
        P = orc.VoLkParams(nlevels=3, min_scale=0, winsize=7, max_iter=21, grad_is_float=1, err_mode=1, gate_on_max_err=1, min_ev=0.01, delta=0.01,
                           max_err=0.6, factor=2.0, pred_div=1.0)
        lk = lambda: o.vo_lk_match_u8(orc.desc_array(prev), orc.desc_array(nxt), orc.desc_array(grad), C.byref(P), kp.ctypes.data, None, n, flow.ctypes.data, dist.ctypes.data)
    s = timed_cpu(lk, share)
    out["pyrlk_1080p_10k"] = {"kpts_per_s": n / s, "kind": cpu.kind, "cores": cpu.threads,
                              "note": "matching only (pyramids prebuilt), pyrlk_match loop with lk_match_point_square_win<7>, vfloat2 gradient"}
    # semi-dense flow 1080p with video_extruder's settings (semi_dense_optical_flow.hpp:46-214: serial by construction, 1 thread)
    g1, g2, _ = scenes.lk_pair(1080, 1920, 4, seed=55, shift=(3.0, -2.0), margin=10)
    h1 = orc.HostImage(1080, 1920, "u8", border=3, aligned=32, data=g1, fill_border="mirror")
    kk = np.zeros((g1.size // 4, 2), dtype=np.int32)
    nk = o.vo_fast9_u8(h1.ptr(), 10, None, 2, 10, 0, kk.ctypes.data, None, len(kk))
    kk = np.ascontiguousarray(kk[:nk])
    i1, i2 = orc.HostImage(1080, 1920, "u8", aligned=32, data=g1), orc.HostImage(1080, 1920, "u8", aligned=32, data=g2)
    rp, rd, rv = np.zeros((nk, 2), np.int32), np.zeros(nk, np.int32), np.zeros(nk, np.uint8)
    sd = (lambda: r.vppref_semi_dense_flow(i1.ptr(), i2.ptr(), kk.ctypes.data, nk, 9, 3, 0, 2, 5, rp.ctypes.data, rd.ctypes.data, rv.ctypes.data)) if r is not None else \
        (lambda: o.vo_semi_dense_flow(i1.ptr(), i2.ptr(), kk.ctypes.data, nk, 9, 3, 0, 2, 5, rp.ctypes.data, rd.ctypes.data, rv.ctypes.data))
    s = timed_cpu(sd, share, max_reps=20)
    out["sdof_1080p"] = {"ms": s * 1e3, "keypoints": int(nk), "kind": cpu.kind, "cores": cpu.threads if r is not None else 1,
                         "note": "pyramids included (the reference builds them inside the call)"}
    return out


# ------------------------------------------------------------------------------------------ GPU arm: shared pieces
def device_ms(torch, dist, dev, fn, reps):
    """CUDA-event time of `reps` calls of fn on the current stream, max over ranks"""
    a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a_.record(torch.cuda.current_stream())
    for _ in range(reps):
        fn()
    b_.record(torch.cuda.current_stream())
    torch.cuda.synchronize()
    t_ = torch.tensor([a_.elapsed_time(b_) / reps], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
    return float(t_.item())


def graph_of(torch, fn):
    """fn replayed as a CUDA graph (same kernels, without the per-launch host cost of the ctypes calls); eager if capture fails"""
    try:
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        g_ = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_):
            fn()
        g_.replay()
        torch.cuda.synchronize()
        return g_.replay, True
    except Exception as ex:  # pragma: no cover
        sys.stderr.write("CUDA graph capture failed, running eagerly: %r\n" % (ex,))
        torch.cuda.synchronize()
        return fn, False


def bind_to_gpu_numa_node(dev_index):
    """One process per GPU: run (and therefore first-touch / pin the host frames of the e2e leg) on the CPUs NVML lists as local to the GPU.
    Returns the number of CPUs bound to, or None when NVML / the affinity call is not available (nothing changes then)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def box_traffic(key):
    """DRAM bytes per launch of the streaming kernel from the committed ncu capture of this bench regime (profiles/box_traffic.json)"""
    tp = os.path.join(ROOT, "profiles", "box_traffic.json")
    if os.path.exists(tp):
        try:
            return json.load(open(tp)).get(key)
        except Exception:
            return None
    return None


def passes_for(ms_per_batch, target_ms=5.5):
    return int(max(1, min(512, np.ceil(target_ms / max(ms_per_batch, 1e-3)))))


def dump_outputs(out_dir, dst, rank, world):
    """The filtered frames the timed step left in this rank's output images (its row tile of each frame at N > 1), as float32
    out_dir/box5x5.npy (box5x5_rank<r>.npy at N > 1) of shape (frames, rows, cols, 3): every row when they fit DUMP_BYTES, else the
    same number of rows of every frame, drawn per frame from a generator seeded with the rank (sorted)."""
    os.makedirs(out_dir, exist_ok=True)
    nrows, ncols = dst[0].nrows, dst[0].ncols
    keep = int(max(1, min(nrows, DUMP_BYTES / world // (len(dst) * ncols * 3 * 4))))
    rng = np.random.default_rng(rank)
    out = np.empty((len(dst), keep, ncols, 3), np.float32)
    for i, d in enumerate(dst):
        out[i] = d.download()[np.sort(rng.choice(nrows, keep, replace=False))]
    np.save(os.path.join(out_dir, "box5x5.npy" if world == 1 else "box5x5_rank%d.npy" % rank), out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=[None] + list(WORKLOADS))
    ap.add_argument("--passes", type=int, default=0, help="launches of the 32-frame batch per step (0 = enough for >= 5 ms of GPU work)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the outputs of the last timed step to DIR/*.npy (float32)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(args.gpus, 1)
    workload = args.workload or ("1080p" if n_gpus == 1 else "8k")
    H, W = WORKLOADS[workload]
    steps, warmup = max(args.steps, 1), max(args.warmup, 3)
    BATCH = BATCH_1GPU if n_gpus == 1 else BATCH_TILED

    base = {"metric": "box5x5_vuchar3_throughput", "unit": "Mpix/s", "n_gpus": n_gpus, "steps": steps, "warmup": warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "5x5 box_filter on %dx%d image2d<vuchar3>%s" % (
                W, H, "" if n_gpus == 1 else ", row-tiled over %d GPUs, halo rows read from the neighbour GPU inside the box kernel (NVLink peer memory)" % n_gpus),
                "frame": [H, W], "resident_frames": BATCH, "border": 2, "row_align": 128,
                "l2": "resident in+out %.0f MB > 126 MB L2, frames cycled" % (2 * BATCH * H * W * 3 / 1e6)}}
    if n_gpus == 1:
        base["config"]["scaling_note"] = ("N=1 is BASELINE configs[1] (1080p); the N>1 lines are strong scaling of the 8K row-tiled workload, whose "
                                          "single-GPU figure is extras.box5x5_vuchar3_8k_x32 (scaling_anchor_n1) of this run")

    if args.impl == "reference":
        if rank != 0:
            return 0
        cb, ms = cpu_box_bench(H, W, steps, warmup, args.cpu_budget)
        line = dict(base)
        line.update({"impl": "reference", "value": cb["value"], "ms_per_step": ms, "cpu_baseline": cb, "gpu_launches": 0,
                     "e2e": {"value": cb["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        line["config"]["frames_per_step"] = int(cb["sample"].split()[0])
        print(json.dumps(line))
        return 0

    import torch

    import vpp_b200 as vpp  # raises when build() has not made vpp_b200/lib/libvppb.so
    from vpp_b200 import capi, tiles
    from tests import oracle as orc  # the checker of what was timed (never the thing measured)

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev_index = local_rank if world > 1 else 0
    numa = bind_to_gpu_numa_node(dev_index) if world > 1 and os.environ.get("VPPB_BENCH_BIND", "0") == "1" else None  # opt-in: no effect measured at N = 2  # pinned host frames then live on the socket the GPU hangs off
    capi.check(capi.lib.vppb_init(dev_index))
    dev = torch.device("cuda", dev_index)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    peak, peak_src = peaks()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- this rank's row tile of every resident frame (the whole frame at N = 1)
    r0, r1 = tiles.tile_rows(H, rank, world)
    th = r1 - r0
    uniq = make_frames(H, W, 4)
    upad = [np.pad(f, ((2, 2), (2, 2), (0, 0)), mode="symmetric") for f in uniq]
    src, dst = [], []
    for i in range(BATCH):
        s = vpp.Image2d(th, W, "vuchar3", border=2)
        blk = np.array(upad[i % 4][r0:r1 + 4])
        if rank > 0:
            blk[:2] = 0xA5   # interior tiles do not hold their halo rows: a broken peer read cannot go unnoticed
        if rank < world - 1:
            blk[-2:] = 0x5A
        s.upload(blk, with_border=True)
        src.append(s)
        dst.append(vpp.Image2d(th, W, "vuchar3"))
    ins = (capi.VppbImg * BATCH)(*[s.desc for s in src])
    outs = (capi.VppbImg * BATCH)(*[d.desc for d in dst])
    opened = []
    if world > 1:
        barrier()
        ups, downs, opened = tiles.open_neighbour_tiles(dist, rank, world, src)
        one_batch = lambda: capi.check(capi.lib.vppb_box5x5_u8c3_tiles(ins, ups, downs, outs, BATCH, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        kernel_name = "k_box5_stream<3,4,0> (tiles: halo rows by bulk copy from peer memory)"
    else:
        one_batch = lambda: capi.check(capi.lib.vppb_box5x5_u8c3_batch(ins, outs, BATCH, C.c_void_p(torch.cuda.current_stream().cuda_stream)))  # the stream current at call time: graph capture runs on a side stream
        kernel_name = "k_box5_stream<3,4,0>"
    one_batch()
    barrier()
    ms_batch = device_ms(torch, dist, dev, one_batch, 10)
    passes = args.passes or passes_for(ms_batch)
    frames_per_step = passes * BATCH
    base["config"].update({"frames_per_step": frames_per_step, "launches_per_step": passes,
                           "step": "%d launches x %d frames (>= 5 ms of GPU work per step)" % (passes, BATCH)})

    def step_eager():
        for _ in range(passes):
            one_batch()

    run_step, graphed = graph_of(torch, step_eager) if args.graph else (step_eager, False)
    base["config"]["cuda_graph"] = graphed
    for _ in range(warmup):
        run_step()
    barrier()
    sampler = ClockSampler(dev_index)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(steps):
        run_step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    if rank == 0 and ms < 400.0 and world == 1:
        t_end = time.perf_counter() + 0.45  # nvidia-smi samples every 100 ms: keep the same load running (untimed) long enough
        while time.perf_counter() < t_end:
            for _ in range(5):
                run_step()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["note"] = "sampled every 100 ms over the timed region" + (" + an untimed continuation of the same step loop" if ms < 400.0 and world == 1 else "")
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    if ms_total / steps < 0.5 * passes * ms_batch:  # a graph that captured nothing would "run" in microseconds
        raise RuntimeError("timed step %.4f ms is far below %d launches x %.4f ms: the step did not execute" % (ms_total / steps, passes, ms_batch))
    value = steps * frames_per_step * H * W / 1e6 / (ms_total / 1e3)

    # ---- parity of what was just timed (frames 0 and BATCH-1, this rank's tile) against the oracle
    hd = []
    for k in (0, (BATCH - 1) % 4):
        hs = orc.HostImage(th, W, "vuchar3", border=2, aligned=32)
        hs.set(upad[k][r0:r1 + 4], with_border=True)
        h_ = orc.HostImage(th, W, "vuchar3", aligned=32)
        orc.load(omp=True).vo_box5x5_u8(hs.ptr(), h_.ptr(), 3)
        hd.append(h_.get())
    parity_ok = bool(np.array_equal(dst[0].download(), hd[0]) and np.array_equal(dst[BATCH - 1].download(), hd[1]))
    if args.dump_outputs:  # every step (timed or the untimed continuation above) writes the same outputs from the same resident inputs
        dump_outputs(args.dump_outputs, dst, rank, world)

    alg_bytes = BOX_BYTES_PER_PX * th * W * BATCH  # per launch, this rank
    us_per_launch = ms_total * 1e3 / (steps * passes)
    achieved = alg_bytes / (us_per_launch * 1e-6) / 1e9
    tkey = "stream_%s_x%d" % (workload, BATCH) if world == 1 else "stream_%s_tile%d_x%d" % (workload, world, BATCH)
    roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": box_traffic(tkey), "peak_source": peak_src, "us_per_launch": us_per_launch, "algorithmic_bytes_per_launch": alg_bytes,
                "how": "6 B/px x %d frames of a launch / (CUDA-event time of the timed region / launches); traffic = dram read + write bytes per launch of the same "
                       "command under ncu (--cache-control none, steady state), profiles/box_traffic.json" % BATCH}

    # ---- e2e: HOST buffers through the C-ABI (pinned), copies inside the timed region, NE2E frames in flight per rank.
    # N > 1: the host holds whole frames, so the 2 halo rows above / below a tile ride along with the tile's upload.
    esets = 8
    if world == 1:
        host_in = [torch.from_numpy(np.ascontiguousarray(uniq[i % 4])).pin_memory() for i in range(4)]
    else:
        host_in = [torch.from_numpy(np.ascontiguousarray(upad[i % 4][r0:r1 + 4])).pin_memory() for i in range(4)]
    host_out = [torch.empty((th, W, 3), dtype=torch.uint8).pin_memory() for _ in range(esets)]
    # frames in flight per rank (one stream each): 12 on one GPU (13.5 k Mpix/s against 12.8 k with 4); with several ranks on one host deeper queues
    # hurt (N = 8: 35.8 k Mpix/s with 12 in flight against 64.2 k with 4; N = 2: 25.5 k against 28.0 k), so 4 there
    NE2E = int(os.environ.get("VPPB_BENCH_INFLIGHT", "12" if world == 1 else "4"))
    e_src = [vpp.Image2d(th, W, "vuchar3", border=2) for _ in range(NE2E)]
    e_dst = [vpp.Image2d(th, W, "vuchar3") for _ in range(NE2E)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(NE2E)]
    rowb = W * 3
    h2d = (th * rowb) if world == 1 else (th + 4) * (W + 4) * 3
    e_frames = min(frames_per_step, 256)  # frames per e2e step (a bounded sample of the step: PCIe time dominates)

    # Two ways to bring a whole host frame into the bordered device image (N = 1), both through the public C-ABI, same launch count:
    #   direct: vppb_upload straight into the pitched image (a 2-D copy: host rows are tight, device rows are padded), then vppb_fill_border_mirror;
    #   staged: vppb_upload into a border-less image whose rows are as tight as the host's (ONE linear copy), then vppb_copy2d_mirror
    #           (copy + mirror border in one launch).  Both are timed; the faster carries the e2e number, both times are reported.
    e_stage = [vpp.Image2d(th, W, "vuchar3") for _ in range(NE2E)] if world == 1 else []
    e2e_mode = ["direct"]

    def e2e_step():
        for i in range(e_frames):
            k = i % NE2E
            st = C.c_void_p(streams[k].cuda_stream)
            hin = host_in[i % len(host_in)]
            if world == 1 and e2e_mode[0] == "staged":
                capi.check(capi.lib.vppb_upload(e_stage[k].ptr(), C.c_void_p(hin.data_ptr()), rowb, 0, st))
                capi.check(capi.lib.vppb_copy2d_mirror(e_stage[k].ptr(), e_src[k].ptr(), st))
            elif world == 1:
                capi.check(capi.lib.vppb_upload(e_src[k].ptr(), C.c_void_p(hin.data_ptr()), rowb, 0, st))
                capi.check(capi.lib.vppb_fill_border_mirror(e_src[k].ptr(), st))
            else:
                origin = hin.data_ptr() + 2 * (W + 4) * 3 + 2 * 3  # pixel (0,0) of the tile inside the padded host rows
                capi.check(capi.lib.vppb_upload(e_src[k].ptr(), C.c_void_p(origin), (W + 4) * 3, 1, st))
            capi.check(capi.lib.vppb_box5x5_u8c3(e_src[k].ptr(), e_dst[k].ptr(), st))
            capi.check(capi.lib.vppb_download(e_dst[k].ptr(), C.c_void_p(host_out[i % esets].data_ptr()), rowb, 0, st))
        for s_ in streams:
            s_.synchronize()

    e2e_ms = {}
    for m_ in (["direct", "staged"] if world == 1 else ["direct"]):
        e2e_mode[0] = m_
        e2e_step()
        torch.cuda.synchronize()
        if not np.array_equal(host_out[0].numpy(), hd[0]):
            sys.stderr.write("e2e form %s gives a different result: not used\n" % m_)
            continue
        t0 = time.perf_counter()
        e2e_step()
        torch.cuda.synchronize()
        e2e_ms[m_] = (time.perf_counter() - t0) * 1e3
    e2e_mode[0] = min(e2e_ms, key=e2e_ms.get) if e2e_ms else "direct"
    for _ in range(2):
        e2e_step()
    barrier()
    esteps = 4
    t0 = time.perf_counter()
    for _ in range(esteps):
        e2e_step()
    torch.cuda.synchronize()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    dt = float(te.item())
    e2e = {"value": esteps * e_frames * H * W / 1e6 / dt, "unit": "Mpix/s", "h2d_bytes_per_step": e_frames * h2d * world,
           "d2h_bytes_per_step": e_frames * th * rowb * world, "ms_per_step": dt / esteps * 1e3, "frames_per_e2e_step": e_frames,
           "upload": {"used": e2e_mode[0], "ms_per_step_by_form": e2e_ms}, "cpus_bound_to_gpu_numa_node": numa,
           "note": "pinned host frames -> vppb_upload (+ mirror border: direct 2-D copy + vppb_fill_border_mirror, or linear copy + vppb_copy2d_mirror, the faster of the two) -> vppb_box5x5_u8c3 -> vppb_download, %d frames in flight per rank, max over ranks" % NE2E}
    parity_ok = parity_ok and bool(np.array_equal(host_out[0].numpy(), hd[0]))
    if dist is not None:  # every rank checked its own tile
        pk = torch.tensor([1.0 if parity_ok else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(pk, op=dist.ReduceOp.MIN)
        parity_ok = bool(pk.item() > 0.5)

    line = dict(base)
    line.update({"value": value, "ms_per_step": ms_total / steps, "clocks": clocks, "roofline": roofline, "e2e": e2e,
                 "gpu_launches": passes * steps, "parity_checked": parity_ok})
    if world > 1:
        # the materialised alternative through the C-ABI, for the record: one grouped NCCL send/recv (vppb_halo_exchange) + plain batch kernel
        try:
            comm = tiles.nccl_comm(dist, rank, world)
            ex = lambda: capi.check(capi.lib.vppb_halo_exchange(comm, rank, world, ins, BATCH, 2, sp))
            plain = lambda: capi.check(capi.lib.vppb_box5x5_u8c3_batch(ins, outs, BATCH, sp))
            ex(); plain()
            torch.cuda.synchronize()
            ok2 = bool(np.array_equal(dst[0].download(), hd[0]))
            line["config"]["nccl_exchange"] = {"exchange_ms_per_launch": device_ms(torch, dist, dev, ex, 10), "exchange_plus_box_ms_per_launch": device_ms(torch, dist, dev, lambda: (ex(), plain()), 10),
                                               "fused_ms_per_launch": ms_batch, "parity": ok2,
                                               "note": "vppb_halo_exchange = ONE grouped NCCL send/recv of the edge rows of all 32 tiles, then the batch kernel; the timed step uses the fused kernel instead"}
            capi.lib.vppb_comm_destroy(comm)
        except Exception as ex_:  # pragma: no cover
            line["config"]["nccl_exchange"] = {"error": repr(ex_)[:200]}

    if world > 1 and not args.no_extras:
        try:
            line.setdefault("extras", {})["sdof_8k_tiled"] = sdof_tiled(vpp, capi, torch, dist, tiles, orc, rank, world, dev, sp)
        except Exception as ex_:  # pragma: no cover
            line.setdefault("extras", {})["sdof_8k_tiled"] = {"error": repr(ex_)[:300]}

    if rank == 0 and n_gpus == 1:
        cb, _ = cpu_box_bench(H, W, 3, 1, args.cpu_budget)
        line["cpu_baseline"] = cb
        if not args.no_extras:
            try:
                line["extras"] = gpu_extras(vpp, capi, torch, stream, sp, dev)
            except Exception as ex:  # pragma: no cover
                line["extras"] = {"error": repr(ex)[:300]}
            try:
                line["extras"]["cpu"] = cpu_extras()
            except Exception as ex:  # pragma: no cover
                line["extras"]["cpu"] = {"error": repr(ex)[:300]}
            a8 = line["extras"].get("box5x5_vuchar3_8k_x32", {})
            if "mpix_per_s" in a8:
                line["scaling_anchor_n1"] = {"value": a8["mpix_per_s"], "unit": "Mpix/s", "workload": "8K vuchar3, 32 frames per launch, one GPU, no tiling",
                                             "hbm_frac": a8.get("hbm_frac")}
    if rank == 0:
        print(json.dumps(line))
    if opened:
        tiles.close_neighbour_tiles(opened)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0 if parity_ok else 3


def sdof_tiled(vpp, capi, torch, dist, tiles, orc, rank, world, dev, sp, H=4320, W=7680, halo=80):
    """BASELINE configs[4]: video_extruder's semi-dense flow on a 7680x4320 frame pair, row-tiled over the ranks.  Every rank owns
    H / world rows of both frames; ONE grouped NCCL halo exchange per frame pair (vppb_halo_exchange, 80 rows each way: SAD window +
    search reach + the 3-level pyramid's footprint, a multiple of patch x 2^(nscales-1) = 20 so that cell grids and pyramid sampling
    line up with the full frame's) extends the tile, then the tile runs the single-GPU path (FAST9 blockwise keypoints of its own rows,
    pyramids, matching, dataflow sweeps).  Semantics are TILE-LOCAL: the propagation sweeps stop at the tile seams, so keypoints near
    a seam may differ from a full-frame run; each rank's result is bit-exact against the oracle on the same extended tile."""
    from tests import scenes
    from vpp_b200.ops import _DeviceBuffer

    g1, g2, _ = scenes.lk_pair(1080, 1920, 4, seed=55, shift=(3.0, -2.0), margin=10)
    g1, g2 = np.tile(g1, (H // 1080, W // 1920)), np.tile(g2, (H // 1080, W // 1920))
    r0, r1 = tiles.tile_rows(H, rank, world)
    th = r1 - r0
    assert th % 20 == 0 and halo % 20 == 0 and halo <= th
    T = [vpp.Image2d(th, W, "u8", border=halo) for _ in range(2)]
    for t_, g in zip(T, (g1, g2)):
        t_.upload(np.ascontiguousarray(g[r0:r1]))
        vpp.fill_border_mirror(t_)          # column borders (and, for the outermost tiles, the frame's own top / bottom)
    comm = tiles.nccl_comm(dist, rank, world)
    descs = (capi.VppbImg * 2)(T[0].desc, T[1].desc)
    top, bot = (halo if rank > 0 else 0), (halo if rank < world - 1 else 0)

    def extended(t_):  # the tile with its halo rows as ordinary domain rows (a view: no copy)
        d = capi.VppbImg()
        C.memmove(C.byref(d), C.byref(t_.desc), C.sizeof(capi.VppbImg))
        d.base = t_.desc.base - top * t_.desc.pitch
        d.alloc = None
        d.nrows = th + top + bot
        d.border = min(3, halo)
        return vpp.Image2d(0, 0, "u8", _desc=d, _owner=t_)

    P = capi.VppbSdofParams(9, 3, 0, 2, 5)
    E = [extended(t_) for t_ in T]
    eh = th + top + bot
    p1, p2 = vpp.Pyramid2d((eh, W), 3, 2, pixel="u8", border=18), vpp.Pyramid2d((eh, W), 3, 2, pixel="u8", border=18)
    wsb = _DeviceBuffer(capi.lib.vppb_sdof_workspace_bytes(eh, W, C.byref(P)))
    capi.check(capi.lib.vppb_halo_exchange(comm, rank, world, descs, 2, halo, sp))
    G = vpp.Image2d(eh, W, "u8", border=3)
    capi.check(capi.lib.vppb_copy2d_mirror(E[0].ptr(), G.ptr(), sp))
    kps = vpp.fast9(G, 10, blockwise=True, block_size=10, stream=sp)
    kps = np.ascontiguousarray(kps[(kps[:, 0] >= top) & (kps[:, 0] < top + th)])  # this rank's own rows
    n = len(kps)
    d_kp = _DeviceBuffer(kps.nbytes).from_host(kps, sp)
    d_pos, d_dist, d_valid = _DeviceBuffer(n * 8), _DeviceBuffer(n * 4), _DeviceBuffer(n)
    a1, a2 = p1.desc_array(), p2.desc_array()

    def frame_pair():
        capi.check(capi.lib.vppb_halo_exchange(comm, rank, world, descs, 2, halo, sp))
        capi.check(capi.lib.vppb_pyrlk_prepare(E[0].ptr(), E[1].ptr(), a1, a2, None, 3, 0, sp))  # both pyramids of the extended tile in one launch
        capi.check(capi.lib.vppb_sdof_u8(a1, a2, C.byref(P), d_kp.ptr, n, wsb.ptr, wsb.nbytes, d_pos.ptr, d_dist.ptr, d_valid.ptr, sp))

    frame_pair()
    got = (d_pos.to_host(np.int32, n * 2, sp).reshape(-1, 2), d_dist.to_host(np.int32, n, sp), d_valid.to_host(np.uint8, n, sp))
    lo, hi = r0 - top, r1 + bot
    h1, h2 = orc.HostImage(eh, W, "u8", data=g1[lo:hi]), orc.HostImage(eh, W, "u8", data=g2[lo:hi])
    rp, rd, rv = np.zeros((n, 2), np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
    orc.load().vo_semi_dense_flow(h1.ptr(), h2.ptr(), kps.ctypes.data, n, 9, 3, 0, 2, 5, rp.ctypes.data, rd.ctypes.data, rv.ctypes.data)
    ok = bool(np.array_equal(got[0], rp) and np.array_equal(got[1], rd) and np.array_equal(got[2], rv))
    ms = device_ms(torch, dist, dev, frame_pair, 5)
    # how far tile-local semantics are from the full-frame flow: every rank runs the oracle on the WHOLE frame pair with the keypoints of all
    # ranks (tiles are bands of whole cells, so their keypoint lists concatenate to the full frame's list) and compares its own rows
    agree = None
    try:
        lists = [None] * world
        dist.all_gather_object(lists, (r0 - top, kps))
        allk = np.ascontiguousarray(np.concatenate([k_ + np.array([off, 0], np.int32) for off, k_ in lists]).astype(np.int32))
        first = int(np.sum([len(k_) for _, k_ in lists[:rank]]))
        m = len(allk)
        fp, fd, fv = np.zeros((m, 2), np.int32), np.zeros(m, np.int32), np.zeros(m, np.uint8)
        F1, F2 = orc.HostImage(H, W, "u8", data=g1), orc.HostImage(H, W, "u8", data=g2)
        orc.load().vo_semi_dense_flow(F1.ptr(), F2.ptr(), allk.ctypes.data, m, 9, 3, 0, 2, 5, fp.ctypes.data, fd.ctypes.data, fv.ctypes.data)
        mine = slice(first, first + n)
        same = (fv[mine] == got[2]) & ((fp[mine] - np.array([r0 - top, 0], np.int32)) == got[0]).all(axis=1) & (fd[mine] == got[1])
        agree = float(same.sum())
    except Exception as ex_:  # pragma: no cover
        agree = None
    tot = torch.tensor([float(n), 1.0 if ok else 0.0, agree if agree is not None else -1e18], dtype=torch.float64, device=dev)
    dist.all_reduce(tot[:1], op=dist.ReduceOp.SUM)
    dist.all_reduce(tot[1:2], op=dist.ReduceOp.MIN)
    dist.all_reduce(tot[2:], op=dist.ReduceOp.SUM)
    capi.lib.vppb_comm_destroy(comm)
    return {"ms_per_frame_pair": ms, "keypoints": int(tot[0].item()), "parity": bool(tot[1].item() > 0.5), "halo_rows": halo,
            "full_frame_agreement": (float(tot[2].item()) / float(tot[0].item())) if tot[2].item() >= 0 and tot[0].item() > 0 else None,
            "note": "NCCL halo exchange (80 rows each way, both frames) + pyramids + matching + sweeps per tile, max over ranks; tile-local semantics, each tile bit-exact "
                    "against the oracle on the same extended tile; full_frame_agreement = fraction of all keypoints whose reported position and distance equal the "
                    "oracle's on the whole frame pair (sweeps do not cross the tile seams); single-GPU anchor: extras.sdof_8k of the N = 1 run"}


def gpu_extras(vpp, capi, torch, stream, sp, dev):
    """Other rows of the hot path, device-resident inputs, CUDA-event timing, each checked against the oracle (`parity`).  Every
    row is measured on its own: one that fails reports {"error": ...} and cannot take the headline line down with it."""
    from tests import oracle as orc, scenes
    from tests.oracle_ops import oracle_grad_pyramid, oracle_lk, oracle_pyramid
    from vpp_b200.ops import _DeviceBuffer

    peak, _ = peaks()
    out = {}
    omp = orc.load(omp=True)

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def add_i32_4k():  # pixel_wise add, 4K int32, 4 triples cycled (398 MB > L2)
        rng = np.random.default_rng(1)
        trip = []
        for _ in range(4):
            b, c = rng.integers(0, 2 ** 30, (2, 2160, 3840), dtype=np.int32)
            trip.append((vpp.Image2d(2160, 3840, "i32"), vpp.Image2d.from_host(b, "i32"), vpp.Image2d.from_host(c, "i32"), b, c))

        def add_all():
            for a_, b_, c_, _, _ in trip:
                capi.check(capi.lib.vppb_pw_add_i32(a_.ptr(), b_.ptr(), c_.ptr(), sp))

        ms = timed(add_all, 20) / len(trip)
        ok = bool(np.array_equal(trip[3][0].download(), trip[3][3] + trip[3][4]))
        return {"mpix_per_s": 2160 * 3840 / 1e6 / (ms / 1e3), "us_per_launch": ms * 1e3, "hbm_frac": 12.0 * 2160 * 3840 / (ms / 1e3) / 1e9 / peak, "parity": ok}

    def box_rows(h, w, nsets, batch):
        f = np.random.default_rng(2).integers(0, 256, (h, w, 3), dtype=np.uint8)
        pairs = []
        for _ in range(nsets):
            s_ = vpp.Image2d.from_host(f, "vuchar3", border=2)
            vpp.fill_border_mirror(s_)
            pairs.append((s_, vpp.Image2d(h, w, "vuchar3")))
        hs = orc.HostImage(h, w, "vuchar3", border=2, aligned=32, data=f, fill_border="mirror")
        hd_ = orc.HostImage(h, w, "vuchar3", aligned=32)
        omp.vo_box5x5_u8(hs.ptr(), hd_.ptr(), 3)
        want = hd_.get()
        if batch:
            n_ = len(pairs)
            bi, bo = (capi.VppbImg * n_)(*[p_[0].desc for p_ in pairs]), (capi.VppbImg * n_)(*[p_[1].desc for p_ in pairs])
            ms = timed(lambda: capi.check(capi.lib.vppb_box5x5_u8c3_batch(bi, bo, n_, sp)), 10) / n_
        else:
            def box_all():
                for s_, d_ in pairs:
                    capi.check(capi.lib.vppb_box5x5_u8c3(s_.ptr(), d_.ptr(), sp))
            ms = timed(box_all, 10) / len(pairs)
        ok = bool(np.array_equal(pairs[-1][1].download(), want) and np.array_equal(pairs[0][1].download(), want))
        return {"mpix_per_s": h * w / 1e6 / (ms / 1e3), "us_per_frame": ms * 1e3, "hbm_frac": 6.0 * h * w / (ms / 1e3) / 1e9 / peak, "parity": ok,
                "launch": "one launch per %d frames" % len(pairs) if batch else "one launch per frame, back to back on one stream"}

    def box5x5_vuchar3_4k():
        return box_rows(2160, 3840, 6, False)

    def box5x5_vuchar3_4k_x16():
        return box_rows(2160, 3840, 16, True)

    def box5x5_vuchar3_8k_x32():  # the N = 1 anchor of the strong-scaling curve: the N > 1 workload on one GPU, no tiling
        return box_rows(4320, 7680, 32, True)

    def ingest_rgb_4k():  # SURVEY 8(f) N1: rgb -> gray + mirror border of 3 in one launch, 4 B/px algorithmic
        f = np.random.default_rng(3).integers(0, 256, (2160, 3840, 3), dtype=np.uint8)
        pairs = [(vpp.Image2d.from_host(f, "vuchar3"), vpp.Image2d(2160, 3840, "u8", border=3)) for _ in range(8)]

        def ingest_all():
            for s_, d_ in pairs:
                capi.check(capi.lib.vppb_rgb_to_graylevel_u8_mirror(s_.ptr(), d_.ptr(), sp))

        ms = timed(ingest_all, 10) / len(pairs)
        exp = np.pad((f.astype(np.int32).sum(axis=2) // 3).astype(np.uint8), 3, mode="symmetric")
        ok = bool(np.array_equal(pairs[0][1].download(with_border=True), exp))
        return {"mpix_per_s": 2160 * 3840 / 1e6 / (ms / 1e3), "us_per_launch": ms * 1e3, "hbm_frac": 4.0 * 2160 * 3840 / (ms / 1e3) / 1e9 / peak, "parity": ok}

    def fast9_4k():
        img = scenes.rectangles_scene(2160, 3840, seed=42)
        G = vpp.Image2d.from_host(img, "u8", border=3)
        vpp.fill_border_mirror(G)
        kps = vpp.fast9(G, 20, stream=sp)
        nk = len(kps)
        hg = orc.HostImage(2160, 3840, "u8", border=3, data=img, fill_border="mirror")
        ref = np.zeros((img.size // 4, 2), dtype=np.int32)
        n_ref = orc.load().vo_fast9_u8(hg.ptr(), 20, None, 0, 10, 0, ref.ctypes.data, None, len(ref))
        ok = bool(n_ref == nk and np.array_equal(kps, ref[:n_ref]))
        from vpp_b200 import ops
        ent = ops._fast_buffers(G, 10, 2160 * 3840 // 8, False)
        run = lambda: capi.check(capi.lib.vppb_fast9_u8_async(G.ptr(), 20, None, 0, 10, 0, ent["ws"].ptr, ent["ws"].nbytes, ent["kps"].ptr, None, ent["cap"], ent["count"].ptr, sp))
        ms_dev = timed(run, 20)
        t0 = time.perf_counter()
        for _ in range(10):
            vpp.fast9(G, 20, stream=sp)
        ms_py = (time.perf_counter() - t0) / 10 * 1e3
        return {"mpix_per_s": 2160 * 3840 / 1e6 / (ms_dev / 1e3), "us_device": ms_dev * 1e3, "hbm_frac": (2160 * 3840 + 8.0 * nk) / (ms_dev / 1e3) / 1e9 / peak,
                "ms_python_call": ms_py, "keypoints": nk, "parity": ok,
                "note": "us_device: detect + raster emit queued by vppb_fast9_u8_async (2 launches, no host sync); ms_python_call adds the count read-back and the keypoint download"}

    def pyrlk_1080p_10k():  # pyramids + Scharr gradient pyramid (vppb_pyrlk_prepare) + pyrlk_match of 10k keypoints, vfloat2 gradient
        f1, f2, pts = scenes.lk_pair(1080, 1920, 10000, seed=5)
        I1, I2 = vpp.Image2d.from_host(f1, "u8"), vpp.Image2d.from_host(f2, "u8")
        prev, nxt = vpp.Pyramid2d((1080, 1920), 3, 2, pixel="u8", border=4), vpp.Pyramid2d((1080, 1920), 3, 2, pixel="u8", border=4)
        grad = vpp.Pyramid2d((1080, 1920), 3, 2, pixel="vfloat2", border=4)
        d_kp = _DeviceBuffer(pts.nbytes).from_host(pts)
        d_flow, d_err = _DeviceBuffer(len(pts) * 8), _DeviceBuffer(len(pts) * 4)
        P = capi.VppbLkParams(nlevels=3, min_scale=0, winsize=7, max_iter=21, grad_is_float=1, err_mode=capi.LK_ERR_SAD_OVER_MAD, gate_on_max_err=1, min_ev=0.01,
                              delta=0.01, max_err=0.6, factor=2.0, pred_div=1.0)
        pa, na, ga = prev.desc_array(), nxt.desc_array(), grad.desc_array()

        def build():
            vpp.pyrlk_prepare(I1, I2, prev, nxt, grad, sp)

        def lk():
            capi.check(capi.lib.vppb_lk_match_u8(pa, na, ga, C.byref(P), d_kp.ptr, None, len(pts), d_flow.ptr, d_err.ptr, sp))

        build(); lk()
        flow, err = d_flow.to_host(np.float32, len(pts) * 2, sp).reshape(-1, 2), d_err.to_host(np.float32, len(pts), sp)
        rprev, rnxt = oracle_pyramid(f1, 3, "u8", 4, omp), oracle_pyramid(f2, 3, "u8", 4, omp)
        rgrad = oracle_grad_pyramid(rprev, "vfloat2", 4, omp)
        RP = orc.VoLkParams(nlevels=3, min_scale=0, winsize=7, max_iter=21, grad_is_float=1, err_mode=1, gate_on_max_err=1, min_ev=0.01, delta=0.01, max_err=0.6,
                            factor=2.0, pred_div=1.0)
        rflow, rerr = oracle_lk(rprev, rnxt, rgrad, RP, pts, lib=omp)
        rel = np.abs(flow - rflow) / np.maximum(np.abs(rflow), 1.0)
        ok = bool(np.array_equal(err >= 3e38, rerr >= 3e38) and (rel <= 1e-4).all())
        ms_build = timed(build, 10)
        ms_lk = timed(lk, 10)
        return {"kpts_per_s": len(pts) / ((ms_lk + ms_build) / 1e3), "kpts_per_s_match_only": len(pts) / (ms_lk / 1e3),
                "ms_match": ms_lk, "ms_pyramids_scharr": ms_build, "parity": ok, "max_rel_err": float(rel.max()),
                "note": "kpts_per_s includes both u8 pyramids and the Scharr gradient pyramid (vppb_pyrlk_prepare: 9 launches, the three independent chains on three streams); parity = failure flags identical and displacement rel. err <= 1e-4 against the oracle "
                        "(whose 3-level definition clamps the reads the reference makes outside its border, tests/test_oracle_vs_ref.py)"}

    def sdof(H_, W_):
        g1, g2, _ = scenes.lk_pair(1080, 1920, 4, seed=55, shift=(3.0, -2.0), margin=10)
        if (H_, W_) != (1080, 1920):  # larger frames: the 1080p pair tiled (the generator's filters take minutes at 8K); same motion everywhere
            g1, g2 = np.ascontiguousarray(np.tile(g1, (H_ // 1080, W_ // 1920))), np.ascontiguousarray(np.tile(g2, (H_ // 1080, W_ // 1920)))
        G = vpp.Image2d.from_host(g1, "u8", border=3)
        vpp.fill_border_mirror(G)
        kps = vpp.fast9(G, 10, blockwise=True, block_size=10, stream=sp)  # video_extruder.hpp:111
        n = len(kps)
        P = capi.VppbSdofParams(9, 3, 0, 2, 5)
        I1, I2 = vpp.Image2d.from_host(g1, "u8"), vpp.Image2d.from_host(g2, "u8")
        p1, p2 = vpp.Pyramid2d(I1, 3, 2, border=18), vpp.Pyramid2d(I2, 3, 2, border=18)
        wsb = _DeviceBuffer(capi.lib.vppb_sdof_workspace_bytes(H_, W_, C.byref(P)))
        d_kp = _DeviceBuffer(kps.nbytes).from_host(kps)
        d_pos, d_dist, d_valid = _DeviceBuffer(n * 8), _DeviceBuffer(n * 4), _DeviceBuffer(n)
        a1, a2 = p1.desc_array(), p2.desc_array()

        def run():
            capi.check(capi.lib.vppb_sdof_u8(a1, a2, C.byref(P), d_kp.ptr, n, wsb.ptr, wsb.nbytes, d_pos.ptr, d_dist.ptr, d_valid.ptr, sp))

        def pyr():  # both pyramids in one launch, as vpp_b200.semi_dense_optical_flow / semi_dense_optical_flow() build them
            capi.check(capi.lib.vppb_pyrlk_prepare(I1.ptr(), I2.ptr(), a1, a2, None, 3, 0, sp))

        run()
        got = (d_pos.to_host(np.int32, n * 2, sp).reshape(-1, 2), d_dist.to_host(np.int32, n, sp), d_valid.to_host(np.uint8, n, sp))
        h1, h2 = orc.HostImage(H_, W_, "u8", data=g1), orc.HostImage(H_, W_, "u8", data=g2)
        rp, rd, rv = np.zeros((n, 2), np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
        k = np.ascontiguousarray(kps)
        orc.load().vo_semi_dense_flow(h1.ptr(), h2.ptr(), k.ctypes.data, n, 9, 3, 0, 2, 5, rp.ctypes.data, rd.ctypes.data, rv.ctypes.data)
        ok = bool(np.array_equal(got[0], rp) and np.array_equal(got[1], rd) and np.array_equal(got[2], rv))
        ms = timed(run, 5)
        ms_pyr = timed(pyr, 5)
        return {"ms": ms + ms_pyr, "ms_flow": ms, "ms_pyramids": ms_pyr, "keypoints": n, "parity": ok,
                "note": "video_extruder's settings (winsize 9, 3 scales, patch 5, 2 sweeps); the whole flow (3 scales: claim, match, sweeps by relaxation, emit) in ONE cooperative launch"}

    def lbp_u8_4k():  # SURVEY 8(f) N4: lbp_transform, 2 B/px algorithmic
        f = np.random.default_rng(4).integers(0, 256, (2160, 3840), dtype=np.uint8)
        pairs = []
        for _ in range(16):  # 16 x (8.3 + 8.3 MB) > L2
            a_ = vpp.Image2d.from_host(f, "u8", border=1)
            vpp.fill_border_mirror(a_)
            pairs.append((a_, vpp.Image2d(2160, 3840, "u8")))

        def lbp_all():
            for s_, d_ in pairs:
                capi.check(capi.lib.vppb_lbp_u8(s_.ptr(), d_.ptr(), sp))

        ms = timed(lbp_all, 10) / len(pairs)
        hs = orc.HostImage(2160, 3840, "u8", border=1, data=f, fill_border="mirror")
        hd_ = orc.HostImage(2160, 3840, "u8")
        orc.load(omp=True).vo_lbp_u8(hs.ptr(), hd_.ptr())
        ok = bool(np.array_equal(pairs[0][1].download(), hd_.get()) and np.array_equal(pairs[-1][1].download(), hd_.get()))
        return {"mpix_per_s": 2160 * 3840 / 1e6 / (ms / 1e3), "us_per_launch": ms * 1e3, "hbm_frac": 2.0 * 2160 * 3840 / (ms / 1e3) / 1e9 / peak, "parity": ok}

    def local_maxima_filter_1080p():  # SURVEY 8(f) N4: in-place filter with the reference's serial semantics, on a FAST-like sparse score image
        r_ = np.random.default_rng(6)
        sc_ = np.where(r_.random((1080, 1920)) < 0.03, r_.integers(1, 250, (1080, 1920)), 0).astype(np.uint8)
        sc_[100:140, 200:900] = (250 - (np.arange(700) % 200))[None, :].astype(np.uint8)  # ramps: chains of dependent decisions
        A_ = vpp.Image2d.from_host(sc_, "u8", border=1)
        vpp.fill_border_with_value(A_, 0)
        src_ = vpp.clone(A_)
        wsb = _DeviceBuffer(capi.lib.vppb_local_maxima_filter_workspace_bytes(1080, 1920, 1))

        def run():
            vpp.copy(src_, A_, sp)
            capi.check(capi.lib.vppb_local_maxima_filter(A_.ptr(), wsb.ptr, wsb.nbytes, sp))

        def copy_only():
            vpp.copy(src_, A_, sp)

        ms = timed(run, 10) - timed(copy_only, 10)
        run()
        hs = orc.HostImage(1080, 1920, "u8", border=1, data=sc_)
        orc.load().vo_local_maxima_filter(hs.ptr())
        ok = bool(np.array_equal(A_.download(), hs.get()))
        return {"mpix_per_s": 1080 * 1920 / 1e6 / (ms / 1e3), "us_per_launch": ms * 1e3, "parity": ok,
                "note": "one cooperative launch: relaxation passes to the fixed point of the serial raster-order filter"}

    def sdof_1080p():
        return sdof(1080, 1920)

    def sdof_8k():  # config 5's kernel on a single GPU: a 7680 x 4320 frame pair
        return sdof(4320, 7680)

    for row in (add_i32_4k, box5x5_vuchar3_4k, box5x5_vuchar3_4k_x16, box5x5_vuchar3_8k_x32, ingest_rgb_4k, fast9_4k, pyrlk_1080p_10k, sdof_1080p, sdof_8k, lbp_u8_4k,
                local_maxima_filter_1080p):
        try:
            out[row.__name__] = row()
        except Exception as ex:  # pragma: no cover - a broken extra must not cost the headline line
            out[row.__name__] = {"error": repr(ex)[:300]}
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
    return out


if __name__ == "__main__":
    sys.exit(main())

"""bench.py's GPU arm executed end to end WITHOUT a GPU (tests/emu/run_bench_emulated.py): the C-ABI calls go to the CPU
emulator and the few torch.cuda pieces the bench uses (streams, events, graphs, device tensors) are replaced by inert
CPU stand-ins.  Nothing is measured here - the point is that every line of the single-GPU control flow (batched launches
per step, graph capture, parity checks against the oracle, roofline / e2e bookkeeping, the reference-kind CPU baseline, the
JSON line) has run before it meets a GPU box, on a tiny geometry.  The N > 1 arm maps the neighbours' tiles through CUDA IPC,
which has no two-process stand-in here: its host logic is covered by tests/test_tiles_gloo.py, its kernels by the
single-process tile test (tests/test_gpu_parity_late.py::test_box5x5_row_tiles_read_neighbours, also emulated) and by
tools/tiles_check.py on real GPUs."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "tests", "emu", "run_bench_emulated.py")
KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
        "roofline", "e2e", "clocks", "gpu_launches", "parity_checked")


def _run(rows, cols, bench_args, env=None):
    return subprocess.Popen([sys.executable, RUNNER, "0", str(rows), str(cols), "--"] + bench_args, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                            text=True, cwd=ROOT, env=env or dict(os.environ))


def test_bench_single_gpu_control_flow(built, tmp_path):
    p = _run(48, 400, ["--steps", "3", "--warmup", "3", "--passes", "2", "--no-extras", "--cpu-budget", "0.2", "--dump-outputs", str(tmp_path)])
    out, err = p.communicate(timeout=900)
    assert p.returncode == 0, err[-3000:]
    line = json.loads(out.strip().splitlines()[-1])
    for key in KEYS + ("cpu_baseline",):
        assert key in line, key
    assert line["parity_checked"] is True
    nb = line["config"]["resident_frames"]
    assert nb == 128 and line["config"]["frames_per_step"] == 2 * nb and line["gpu_launches"] == 3 * 2
    assert line["roofline"]["algorithmic_bytes_per_launch"] == 6.0 * 48 * 400 * nb
    ef = line["e2e"]["frames_per_e2e_step"]
    assert line["e2e"]["h2d_bytes_per_step"] == ef * 48 * 400 * 3 and line["e2e"]["d2h_bytes_per_step"] == ef * 48 * 400 * 3
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    # --dump-outputs: at this size every row of the 128 output frames fits; frame i is the box filter of seeded input i % 4
    from bench import make_frames
    from tests import oracle as orc

    assert os.listdir(str(tmp_path)) == ["box5x5.npy"]
    out = np.load(str(tmp_path / "box5x5.npy"))
    assert out.dtype == np.float32 and out.shape == (nb, 48, 400, 3)
    for i, f in enumerate(make_frames(48, 400, 4)):
        hs = orc.HostImage(48, 400, "vuchar3", border=2, data=f, fill_border="mirror")
        hd = orc.HostImage(48, 400, "vuchar3")
        orc.load().vo_box5x5_u8(hs.ptr(), hd.ptr(), 3)
        assert np.array_equal(out[i::4], np.broadcast_to(hd.get(), out[i::4].shape)), i


def test_bench_reference_arm(built):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-budget", "0.5"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]

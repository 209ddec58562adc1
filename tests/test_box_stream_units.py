"""The work units of the streaming box kernel on the CPU emulator: a warp takes 4 consecutive units of 128 output bytes x R rows
in (image, row chunk, column unit) order, so its units may end a row chunk, start the next one or the next image, and the last
task of a launch may hold fewer than 4.  Widths put the byte rows just before, on and after a multiple of 128 bytes (a lane
partly or wholly right of the image); row counts leave a short last chunk; image counts leave a partial last task."""
import numpy as np
import pytest

from tests.test_emulated_property import _box_oracle, vpp  # noqa: F401  (the module-scoped emulator fixture)

CASES = [
    # pix, rows, cols, images: byte rows 381 / 384 / 387 (vuchar3), 127 / 128 / 129 and 255 / 256 / 257 (u8)
    ("vuchar3", 21, 127, 3),
    ("vuchar3", 21, 128, 3),
    ("vuchar3", 21, 129, 3),
    ("u8", 17, 127, 5),
    ("u8", 17, 128, 5),
    ("u8", 17, 129, 5),
    ("u8", 40, 255, 3),
    ("u8", 40, 256, 2),
    ("u8", 40, 257, 3),
    # one unit per row chunk: every warp's 4 units lie in 4 different chunks, and cross into the next image
    ("u8", 45, 100, 3),
    # 5 units per row: warps straddle row chunks; 33 rows = a short last chunk
    ("vuchar3", 33, 213, 2),
    # 2 rows: a chunk shorter than the first stage's window
    ("vuchar3", 2, 300, 7),
]


@pytest.mark.parametrize("pix,nr,nc,n", CASES)
def test_box_stream_units(vpp, pix, nr, nc, n):  # noqa: F811
    ch = 3 if pix == "vuchar3" else 1
    r = np.random.default_rng(nr * 1000 + nc)
    frames = [r.integers(0, 256, (nr, nc) + ((ch,) if ch > 1 else ()), dtype=np.uint8) for _ in range(n)]
    srcs, dsts = [], []
    for f in frames:
        S = vpp.Image2d.from_host(f, pix, border=2)
        vpp.fill_border_mirror(S)
        srcs.append(S)
        dsts.append(vpp.Image2d(nr, nc, pix))
    vpp.box5x5_batch(srcs, dsts)
    for i, f in enumerate(frames):
        assert np.array_equal(dsts[i].download(), _box_oracle(f, pix)), (i, nr, nc, n)

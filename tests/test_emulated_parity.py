"""The `-m gpu` parity tests of tests/test_gpu_parity.py, run a second time WITHOUT a GPU: the same Python host code
(vpp_b200.ops / image / video_extruder) drives tests/emu/_build/libvppb_emu.so — the library's own .cu sources
(core, pixelwise, pyramid, colorspace, box, fast, lk, sdof) compiled by g++ and executed by the fiber-per-thread block/warp emulator
of tests/emu/ — and every result is compared with the oracle exactly as on the GPU.

This checks the kernels' logic (indexing, warp collectives, barriers, atomics' results, float evaluation order) and
the host-side orchestration on the CPU.  It says nothing about speed, and it does not cover what only the hardware
can show (the real TMA unit and mbarrier hardware — tests/emu/tma.cuh only models their documented behaviour and alignment
rules —, memory-model races between concurrently running blocks).
TEST INFRASTRUCTURE: the emulated library is never loaded by the product path."""
import ctypes as C
import gc
import glob
import os
import sys

import pytest

from tests import test_gpu_parity as G
from tests import test_gpu_parity_late as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UBSAN_LOG = os.path.join(ROOT, "tests", "emu", "_build", "ubsan.log")


SCHEDULES = os.environ.get("VPPB_EMU_SCHEDULES", "forward,shuffled").split(",")  # "forward,reversed,shuffled" for all three


@pytest.fixture(scope="module", params=SCHEDULES)
def vpp(built, request):
    """`reversed`: blocks and the threads inside a block are scheduled last to first - a result that depends on which
    thread / block gets somewhere first (an unordered atomic append, a missing barrier) changes and fails the comparison;
    `shuffled`: every scheduler round visits the threads of the block in a fresh pseudo-random order (seeded)"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu

    path = build_emu.build(asan=os.environ.get("VPPB_EMU_ASAN") == "1")  # the ASan variant needs libasan preloaded (tests/test_emulated_asan.py)
    for f in glob.glob(UBSAN_LOG + "*"):
        os.remove(f)
    os.environ.setdefault("UBSAN_OPTIONS", "log_path=%s" % UBSAN_LOG)  # same path as tests/test_emulated_kernels.py: the .so is loaded once per process
    os.environ.setdefault("VPPB_EMU_LOG", os.path.join(ROOT, "tests", "emu", "_build", "emu_fail.log"))  # why the emulator aborted, if it does
    emu = C.CDLL(path)
    import vpp_b200
    from vpp_b200 import capi, ops

    for name, (res, args) in capi.PROTOTYPES.items():
        fn = getattr(emu, name)
        fn.restype, fn.argtypes = res, args
    emu.vppb_emu_set_reverse(1 if request.param == "reversed" else 0)
    emu.vppb_emu_set_shuffle(12345 if request.param == "shuffled" else 0)
    # ops caches FAST workspaces across calls: a cached buffer must be freed by the library that allocated it and never reach
    # the other one (emulator buffers are host memory; freeing one with cudaFree leaves an error pending in the CUDA runtime)
    ops._FAST_CACHE.clear()
    mp = pytest.MonkeyPatch()
    mp.setattr(capi, "lib", emu)
    mp.setattr(ops, "lib", emu)
    yield vpp_b200
    emu.vppb_emu_set_reverse(0)
    emu.vppb_emu_set_shuffle(0)
    ops._FAST_CACHE.clear()
    gc.collect()  # images allocated by the emulated library must be freed by it
    mp.undo()
    logs = glob.glob(UBSAN_LOG + "*")
    text = "".join(open(f).read() for f in logs)
    assert not text, "UBSan reports from the emulated kernels:\n" + text[:4000]


# containers, maps, fills, copies, sum (warp shuffle reduction + atomicAdd)
test_layout_alignment_and_roundtrip = G.test_layout_alignment_and_roundtrip
test_subimage_aliases_pixels = G.test_subimage_aliases_pixels
test_pixel_wise_add_bit_exact = G.test_pixel_wise_add_bit_exact
test_pixel_wise_add_wraps_and_views = G.test_pixel_wise_add_wraps_and_views
test_fill_variants = G.test_fill_variants
test_border_fills = G.test_border_fills
test_border_closest_closed_form = G.test_border_closest_closed_form
test_copy_clone_sum = G.test_copy_clone_sum
# 5x5 box: the persistent two-phase tile kernel with its TMA loads and mbarrier emulated (tests/emu/tma.cuh asserts the
# alignment rules the hardware enforces), and the direct kernel used for views / small alignments
test_box5x5_vuchar3_bit_exact = G.test_box5x5_vuchar3_bit_exact
test_box5x5_extremes_and_u8 = G.test_box5x5_extremes_and_u8
test_box5x5_direct_path_on_views_matches = G.test_box5x5_direct_path_on_views_matches
test_box5x5_i32 = G.test_box5x5_i32
test_box5x5_batch_equals_oracle = L.test_box5x5_batch_equals_oracle
test_box5x5_batch_fallbacks_and_errors = L.test_box5x5_batch_fallbacks_and_errors
test_box_border_too_small_is_an_error = G.test_box_border_too_small_is_an_error
# frame ingest (rgb_to_graylevel, fused with the mirror border)
test_rgb_to_graylevel_and_frame_ingest = L.test_rgb_to_graylevel_and_frame_ingest
# Scharr, pyramids (fused level launches)
test_scharr = G.test_scharr
test_pyramid_u8 = G.test_pyramid_u8
test_gradient_pyramid = G.test_gradient_pyramid
test_fused_level_equals_lowpass_then_mirror = L.test_fused_level_equals_lowpass_then_mirror
# FAST9 (ballots, block scans, atomics), Lucas-Kanade (4 keypoints per warp, ordered float sums), semi-dense flow
test_fast9_keypoints_bit_exact = G.test_fast9_keypoints_bit_exact
test_fast9_mask_semantics = G.test_fast9_mask_semantics
test_fast9_maxima_modes = G.test_fast9_maxima_modes
test_fast9_edges_empty_and_errors = G.test_fast9_edges_empty_and_errors
test_lucas_kanade_driver = G.test_lucas_kanade_driver
test_lucas_kanade_prediction_and_failures = G.test_lucas_kanade_prediction_and_failures
test_pyrlk_match = G.test_pyrlk_match
test_halo_pack_unpack_single_and_batch = G.test_halo_pack_unpack_single_and_batch
test_semi_dense_optical_flow_bit_exact = G.test_semi_dense_optical_flow_bit_exact
test_video_extruder_gpu_equals_oracle = G.test_video_extruder_gpu_equals_oracle
test_video_extruder_eventful_sequence_equals_reference_tables = L.test_video_extruder_eventful_sequence_equals_reference_tables
test_linear_copy_path_of_upload_download = L.test_linear_copy_path_of_upload_download
test_semi_dense_flow_level_schedule = L.test_semi_dense_flow_level_schedule
test_semi_dense_flow_long_propagation_chains = L.test_semi_dense_flow_long_propagation_chains
test_pyrlk_prepare_one_launch_equals_streams = L.test_pyrlk_prepare_one_launch_equals_streams
test_fast9_wide_images_multibox = L.test_fast9_wide_images_multibox
test_fast9_threshold_extremes = L.test_fast9_threshold_extremes
test_box5x5_row_tiles_read_neighbours = L.test_box5x5_row_tiles_read_neighbours
test_video_extruder_device_container_equals_reference_tables = L.test_video_extruder_device_container_equals_reference_tables
test_video_extruder_device_container_merge_cases = L.test_video_extruder_device_container_merge_cases
test_out_of_frame_keypoints_are_skipped = L.test_out_of_frame_keypoints_are_skipped

# SURVEY 8(f) N4: lbp_transform, local_maxima_filter (cooperative relaxation kernel on a grid of one block), blockwise_rank, oriented LK
from tests import test_gpu_n4 as N4  # noqa: E402

test_lbp_transform = N4.test_lbp_transform
test_local_maxima_filter_serial_semantics = N4.test_local_maxima_filter_serial_semantics
test_fast9_blockwise_rank = N4.test_fast9_blockwise_rank
test_oriented_lk_matcher = N4.test_oriented_lk_matcher

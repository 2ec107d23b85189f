"""The launch plan of a call of several views (lt_debug_plan_views, no device needed) and the argument checks of the views
entry points.  Device: 180 GiB and 148 SMs (a B200); scenes as in test_launch_plan.py."""
import ctypes as C

import numpy as np
import pytest

from lens_trace_b200 import capi, layouts as L
from lens_trace_b200.capi import PIPE_PATH, PIPE_WAVEFRONT

B200 = dict(total_mem=180 << 30, sm_count=148)
SMALL = dict(node_count=83, stack_depth=8)
LARGE = dict(node_count=1999419, stack_depth=40)
HUGE = dict(node_count=20000000, stack_depth=40)

KERNELS = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY, L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR,
           L.KERNEL_GI25, L.KERNEL_GI]
FLAGS = [0, L.FLAG_STATS, L.FLAG_STATS | L.FLAG_STATS_TRACED, L.FLAG_CULL, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT,
         L.FLAG_SERIAL, L.FLAG_NO_THREADED, L.FLAG_NO_STREAM]
SIZES = [(101, 75), (1920, 1080), (3840, 2160)]


def plans(params, views, scene=SMALL):
    return capi.plan_views(params, views, scene["node_count"], scene["stack_depth"], B200["total_mem"],
                           B200["sm_count"])


@pytest.mark.parametrize("scene", [SMALL, LARGE, HUGE])
@pytest.mark.parametrize("kernel", KERNELS)
def test_one_view_is_the_single_plan(kernel, scene):
    for w, h in SIZES:
        for frames in (1, 4, 5, 64):
            for flags in FLAGS:
                for depth in (0, 4, 40):
                    p = capi.make_params(kernel, w, h, frames=frames, flags=flags, max_ray_depth=depth)
                    want = capi.plan(p, scene["node_count"], scene["stack_depth"], B200["total_mem"],
                                     B200["sm_count"])
                    assert plans(p, 1, scene) == want, (w, h, frames, flags, depth)


def test_views_move_one_frame_gi_to_the_wavefront():
    """1080p GI, one frame per view: the views' paths count together (2 073 600 per view); views take the wavefront from
    3 * 2^20 paths, between the measured crossover points of one view (megakernel faster) and two (wavefront faster)"""
    p = capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=4)
    assert plans(p, 1)["pipeline"] == PIPE_PATH
    for v in (2, 4, 8, 16, 64):
        got = plans(p, v)
        assert got["error"] == 0 and got["pipeline"] == PIPE_WAVEFRONT, v
        assert got["shared_primary"] == 1 and got["classify"] == 1 and got["streams"] == 2
    # a batch holds at most 2^25 paths and, both overlapped batches together, 2^26: 16 views of 1080p, 8 per batch
    assert plans(p, 16)["batch_frames"] == 8
    # below the threshold: two 720p views (1 843 200 paths) stay on the megakernel, three (2 764 800) too, four go
    p.width, p.height = 1280, 720
    assert plans(p, 2)["pipeline"] == PIPE_PATH
    assert plans(p, 3)["pipeline"] == PIPE_PATH
    assert plans(p, 4)["pipeline"] == PIPE_WAVEFRONT
    # the 25-sample kernels stay on the megakernel, as for frames
    p.kernel = L.KERNEL_GI25
    assert plans(p, 64)["pipeline"] == PIPE_PATH


def test_views_and_frames_count_together():
    p = capi.make_params(L.KERNEL_GI, 960, 540, frames=2, max_ray_depth=4)
    assert plans(p, 2)["pipeline"] == PIPE_PATH  # 4 pairs, 2 073 600 paths
    got = plans(p, 4)  # 8 pairs, 4 147 200 paths
    assert got["pipeline"] == PIPE_WAVEFRONT and got["batch_frames"] == 4


def test_workspace_bound_for_1024_views_of_4k():
    """the primary records cover the views one batch touches, not all views of the call"""
    w, h = 3840, 2160
    pixels = w * h
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4)
    got = plans(p, 1024)
    assert got["pipeline"] == PIPE_WAVEFRONT
    b, streams = got["batch_frames"], got["streams"]
    assert (b, streams) == (4, 2)
    single = capi.plan(capi.make_params(L.KERNEL_GI, w, h, frames=8, max_ray_depth=4), **SMALL, **B200)
    queues = single["workspace_bytes"] - (29 * pixels + 1024 + 5 * 256)  # the same two batch workspaces
    record = (29 * pixels + 1024 + 5 * 256 + 255) // 256 * 256
    assert got["workspace_bytes"] == queues + streams * b * record  # one view per pair of a one-frame batch
    assert got["workspace_bytes"] < 2 * single["workspace_bytes"]
    # several frames per view: a batch touches at most (frames + batch - 2) // frames + 1 views
    p.frames = 3
    got = plans(p, 1024)
    b = got["batch_frames"]
    touched = min(1024, (3 + b - 2) // 3 + 1)
    assert got["workspace_bytes"] - queues == streams * touched * record


def test_plan_with_a_batch_boundary_inside_a_view():
    """3 views x 3 frames on two streams: batches of 5 (view, frame) pairs; the first batch ends inside view 1 and the
    9 pairs are not a multiple of the batch (tests/test_gpu_views.py renders this plan)"""
    p = capi.make_params(L.KERNEL_GI, 128, 96, max_ray_depth=4, frames=3, accum_mode=L.ACCUM_RUNNING_MEAN,
                         flags=L.FLAG_WAVEFRONT)
    got = plans(p, 3)
    assert got["pipeline"] == PIPE_WAVEFRONT and got["batch_frames"] == 5 and got["streams"] == 2
    assert 3 % 5 != 0 and (3 * 3) % 5 != 0


def test_stats_and_cull_views_keep_no_primary_records():
    p = capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=4, flags=L.FLAG_STATS)
    got = plans(p, 8)
    assert got["pipeline"] == PIPE_WAVEFRONT and got["shared_primary"] == 0 and got["streams"] == 1
    assert got["workspace_bytes"] == plans(capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=4, frames=8,
                                                            flags=L.FLAG_STATS), 1)["workspace_bytes"] - (
        29 * 1920 * 1080 + 1024 + 5 * 256)


def test_argument_errors_without_a_device():
    lib = capi.load()
    p = capi.make_params(L.KERNEL_GI, 64, 64)
    out = (C.c_int64 * len(capi.PLAN_FIELDS))()
    assert lib.lt_debug_plan_views(C.byref(p), 0, 83, 8, B200["total_mem"], B200["sm_count"], out) == capi.ERR_INVALID
    assert lib.lt_debug_plan_views(C.byref(p), -3, 83, 8, B200["total_mem"], B200["sm_count"], out) == capi.ERR_INVALID
    cams = np.concatenate([L.make_camera(0, 2.5, -50, 0.0, k) for k in range(3)])
    # the view count and the cameras are checked before the context: no device is needed to see these errors
    assert lib.lt_render_views(None, None, cams.ctypes.data, 0, C.byref(p), None) == capi.ERR_INVALID
    assert b"view_count" in lib.lt_last_error(None)
    assert lib.lt_render_views(None, None, None, 3, C.byref(p), None) == capi.ERR_INVALID
    assert b"cameras28" in lib.lt_last_error(None)
    assert lib.lt_render_views_device(None, None, cams.ctypes.data, 0, C.byref(p), None, 1) == capi.ERR_INVALID
    assert lib.lt_render_views_device(None, None, None, 3, C.byref(p), None, 1) == capi.ERR_INVALID
    assert lib.lt_render_views(None, None, cams.ctypes.data, 3, C.byref(p), None) == capi.ERR_INVALID
    assert b"ctx is NULL" in lib.lt_last_error(None)

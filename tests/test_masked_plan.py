"""The launch plan of a masked call (lt_debug_plan_masked, no device needed): every size counts the listed pixels, a full
mask plans as the unmasked call, and the deterministic kernels run k_flat over the list.  Device: 180 GiB and 148 SMs (a
B200); scenes as in test_launch_plan.py."""
import ctypes as C

import pytest

from lens_trace_b200 import capi, layouts as L
from lens_trace_b200.capi import PIPE_FLAT, PIPE_FLAT_STREAM, PIPE_PATH, PIPE_WAVEFRONT

B200 = dict(total_mem=180 << 30, sm_count=148)
SMALL = dict(node_count=83, stack_depth=8)
LARGE = dict(node_count=1999419, stack_depth=40)

KERNELS = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY, L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR,
           L.KERNEL_GI25, L.KERNEL_GI]
DETERMINISTIC = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY]
FLAGS = [0, L.FLAG_STATS, L.FLAG_STATS | L.FLAG_STATS_TRACED, L.FLAG_CULL, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT,
         L.FLAG_SERIAL, L.FLAG_NO_THREADED, L.FLAG_NO_STREAM]
SIZES = [(101, 75), (128, 96), (1920, 1080), (3840, 2160)]


def masked(params, n, scene=SMALL):
    return capi.plan_masked(params, n, scene["node_count"], scene["stack_depth"], B200["total_mem"], B200["sm_count"])


def single(params, scene=SMALL):
    return capi.plan(params, scene["node_count"], scene["stack_depth"], B200["total_mem"], B200["sm_count"])


@pytest.mark.parametrize("kernel", KERNELS)
def test_full_mask_is_the_unmasked_plan(kernel):
    for w, h in SIZES:
        for frames in (1, 4, 64):
            for flags in FLAGS:
                for depth in (0, 4, 40):
                    p = capi.make_params(kernel, w, h, frames=frames, flags=flags, max_ray_depth=depth)
                    assert masked(p, w * h) == single(p), (w, h, frames, flags, depth)


@pytest.mark.parametrize("kernel", [L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR, L.KERNEL_GI25, L.KERNEL_GI])
def test_full_mask_on_a_large_scene(kernel):
    """the stochastic kernels on the large-scene tree choice plan as unmasked there too"""
    for w, h in SIZES:
        for flags in FLAGS:
            p = capi.make_params(kernel, w, h, frames=16, flags=flags, max_ray_depth=4)
            assert masked(p, w * h, LARGE) == single(p, LARGE), (w, h, flags)


def test_partial_gi_lists_take_the_wavefront_at_the_measured_thresholds():
    """scattered pixels: a partial GI list takes the wavefront from 2^20 paths, and from 2^16 paths at 16 frames or more
    (measured, tools/masked_timing.py); fewer paths stay on the megakernel, as does a full list below the image's 2^23"""
    w, h = 1920, 1080
    p = capi.make_params(L.KERNEL_GI, w, h, frames=1, max_ray_depth=4)
    assert single(p)["pipeline"] == PIPE_PATH and masked(p, w * h)["pipeline"] == PIPE_PATH
    assert masked(p, w * h - 1)["pipeline"] == PIPE_WAVEFRONT
    assert masked(p, 1 << 20)["pipeline"] == PIPE_WAVEFRONT
    few = masked(p, (1 << 20) - 1)
    assert few["pipeline"] == PIPE_PATH and few["grid"] == ((1 << 20) - 1 + 127) // 128
    p.frames = 4
    assert masked(p, 1 << 18)["pipeline"] == PIPE_WAVEFRONT
    assert masked(p, (1 << 18) - 1)["pipeline"] == PIPE_PATH
    for frames in (16, 64):
        p.frames = frames
        assert masked(p, (1 << 16) // frames)["pipeline"] == PIPE_WAVEFRONT
        assert masked(p, (1 << 16) // frames - 1)["pipeline"] == PIPE_PATH
    p.frames = 15  # below 16 frames only the 2^20 paths count
    assert masked(p, 1 << 16)["pipeline"] == PIPE_PATH  # 983 040 paths
    assert masked(p, 69906)["pipeline"] == PIPE_WAVEFRONT  # 1 048 590 paths
    # LT_FLAG_MEGAKERNEL keeps the megakernel; the other kernels keep the image's thresholds (not measured for lists)
    p.flags = L.FLAG_MEGAKERNEL
    assert masked(p, 1 << 20)["pipeline"] == PIPE_PATH
    for kernel in (L.KERNEL_ACCUMULATOR, L.KERNEL_LIGHTING25, L.KERNEL_GI25):
        q = capi.make_params(kernel, w, h, frames=16, max_ray_depth=4)
        for n in (1 << 16, 1 << 20):
            want = single(capi.make_params(kernel, n, 1, frames=16, max_ray_depth=4))["pipeline"]
            assert masked(q, n)["pipeline"] == want, (kernel, n)



def test_wavefront_sizes_follow_the_list():
    """frames per batch, workspace and primary records are those of an image of N pixels"""
    w, h = 3840, 2160
    for n in (w * h // 2, 1 << 20, 12345):
        p = capi.make_params(L.KERNEL_GI, w, h, frames=64, max_ray_depth=4, flags=L.FLAG_WAVEFRONT)
        got = masked(p, n)
        # the same call on an image of n pixels (one row of n) plans the same sizes
        want = single(capi.make_params(L.KERNEL_GI, n, 1, frames=64, max_ray_depth=4, flags=L.FLAG_WAVEFRONT))
        assert got["pipeline"] == PIPE_WAVEFRONT
        for k in ("batch_frames", "streams", "rounds", "workspace_bytes", "grid", "shared_primary", "classify"):
            assert got[k] == want[k], (n, k)
    big = masked(capi.make_params(L.KERNEL_GI, w, h, frames=64, max_ray_depth=4), 1 << 20)
    assert big["batch_frames"] > single(capi.make_params(L.KERNEL_GI, w, h, frames=64, max_ray_depth=4))["batch_frames"]


@pytest.mark.parametrize("kernel", DETERMINISTIC)
def test_deterministic_kernels_run_k_flat(kernel):
    """never k_flat_stream, which fetches whole pixel tiles: k_flat over the list, one thread per listed pixel"""
    w, h = 1920, 1080
    p = capi.make_params(kernel, w, h)
    assert single(p, LARGE)["pipeline"] == PIPE_FLAT_STREAM
    for n in (w * h, w * h // 3, 1):
        got = masked(p, n, LARGE)
        assert got["pipeline"] == PIPE_FLAT and got["tree"] == single(p, LARGE)["tree"], n
        assert got["grid"] == (single(capi.make_params(kernel, w, h, flags=L.FLAG_NO_STREAM), LARGE)["grid"]
                               if n == w * h else (n + 127) // 128)
    for flags in FLAGS:
        p.flags = flags
        assert masked(p, 1000, SMALL)["pipeline"] == PIPE_FLAT


def test_path_limit_and_forced_errors_follow_the_list():
    """the wavefront holds at most 2^25 paths per frame: of listed pixels, not of the image's"""
    w, h = 8192, 8192  # 2^26 pixels
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, flags=L.FLAG_WAVEFRONT)
    assert single(p)["error"] == capi.ERR_UNSUPPORTED
    assert masked(p, w * h)["error"] == capi.ERR_UNSUPPORTED
    assert "2^25" in masked(p, (1 << 25) + 1)["message"]
    got = masked(p, 1 << 25)
    assert got["error"] == 0 and got["pipeline"] == PIPE_WAVEFRONT and got["batch_frames"] == 1
    # the default schedule keeps such a call on the megakernel instead of failing
    p.flags = 0
    p.frames = 4
    assert masked(p, w * h)["pipeline"] == PIPE_PATH and masked(p, w * h)["error"] == 0
    assert masked(p, 1 << 24)["pipeline"] == PIPE_WAVEFRONT
    # a bounce cap the wavefront cannot carry: the same error for any list
    p = capi.make_params(L.KERNEL_GI, 64, 64, max_ray_depth=40, flags=L.FLAG_WAVEFRONT)
    assert masked(p, 10)["error"] == capi.ERR_UNSUPPORTED


def test_images_above_int_max_pixels_are_refused():
    """the pixel list holds 32-bit pixel indices: an image of more than 2^31 - 1 pixels is LT_ERR_UNSUPPORTED (the
    unmasked call still plans it, on the megakernel)"""
    for w, h in ((50000, 50000), (46341, 46341), (65536, 32768)):
        p = capi.make_params(L.KERNEL_GI, w, h)
        assert single(p)["error"] == 0
        for n in (1, 1000, (1 << 31) - 1):
            got = masked(p, n)
            assert got["error"] == capi.ERR_UNSUPPORTED and "2^31 - 1 pixels" in got["message"], (w, h, n)
    p = capi.make_params(L.KERNEL_GI, 46340, 46340)  # 2 147 395 600 pixels: the largest square image that fits
    got = masked(p, 46340 * 46340)
    assert got["error"] == 0 and got["pipeline"] == PIPE_PATH and got["grid"] == single(p)["grid"]
    got = masked(p, (1 << 31) - 200000)
    assert got["error"] == 0 and got["grid"] == ((1 << 31) - 200000 + 127) // 128


def test_argument_errors_without_a_device():
    lib = capi.load()
    p = capi.make_params(L.KERNEL_GI, 64, 64)
    out = (C.c_int64 * len(capi.PLAN_FIELDS))()
    for n in (0, -1, 64 * 64 + 1):
        assert lib.lt_debug_plan_masked(C.byref(p), n, 83, 8, B200["total_mem"], B200["sm_count"], out) == \
            capi.ERR_INVALID, n
    with pytest.raises(capi.LtError):
        masked(p, 0)
    bad = capi.make_params(L.KERNEL_GI, 0, 64)
    assert lib.lt_debug_plan_masked(C.byref(bad), 1, 83, 8, B200["total_mem"], B200["sm_count"], out) == \
        capi.ERR_INVALID
    assert lib.lt_render_masked_device(None, None, None, C.byref(p), None, None, None, 1) == capi.ERR_INVALID
    assert b"ctx is NULL" in lib.lt_last_error(None)

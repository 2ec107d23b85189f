"""Adaptive sampling without a device: the round schedule of lt_render_adaptive (lt_debug_adaptive_rounds), its argument
errors with their codes and messages, the NULL-context checks, the scene-file keys that reach RenderExtensionB200, and
the row partition the devices of a multi-GPU context share."""
import ctypes as C
import json

import numpy as np
import pytest

from lens_trace_b200 import capi, host, layouts as L

W, H = 101, 75


def params(frames=16, **kw):
    kw.setdefault("accum_mode", L.ACCUM_RUNNING_MEAN)
    return capi.make_params(L.KERNEL_GI, W, H, max_ray_depth=4, frames=frames, **kw)


def rounds(frames, max_frames, round_frames=0, first=0, target=0.05):
    return capi.adaptive_rounds(params(frames), capi.make_adaptive(target, max_frames, round_frames), first)


def test_round_schedule():
    assert rounds(16, 64) == [16, 16, 16, 16]                 # round_frames 0: params.frames
    assert rounds(16, 64, round_frames=8) == [16] + [8] * 6
    assert rounds(16, 40, round_frames=10) == [16, 10, 10, 4]  # the last round clipped to max_frames
    assert rounds(16, 16) == [16]                             # max_frames == frames: one round
    assert rounds(2, 3, round_frames=5) == [2, 1]
    assert rounds(1, 4, round_frames=1, first=1) == [1, 1, 1, 1]  # continuation: frameCount 1 + 1 frame
    assert rounds(4, 12, first=100) == [4, 4, 4]               # the schedule counts this call's frames only


def error_of(p, a, first=0):
    with pytest.raises(capi.LtError) as e:
        capi.adaptive_rounds(p, a, first)
    return e.value.code, str(e.value).split(": ", 1)[1]


def test_argument_errors():
    good = capi.make_adaptive(0.05, 64)
    inv, uns = capi.ERR_INVALID, capi.ERR_UNSUPPORTED
    need_mean = "lt_render_adaptive: needs accum_mode LT_ACCUM_RUNNING_MEAN and frame_stride <= 1"
    assert error_of(params(accum_mode=L.ACCUM_NONE), good) == (inv, need_mean)
    assert error_of(params(accum_mode=L.ACCUM_WEIGHTED_SUM), good) == (inv, need_mean)
    assert error_of(params(frame_stride=2), good) == (inv, need_mean)
    two = "lt_render_adaptive: camera.frameCount + frames must be >= 2 (a variance needs two frames)"
    assert error_of(params(frames=1), capi.make_adaptive(0.05, 4)) == (inv, two)
    assert capi.adaptive_rounds(params(frames=1), capi.make_adaptive(0.05, 4), 1) == [1, 1, 1, 1]
    target = "lt_render_adaptive: target must be finite and > 0"
    for t in (0.0, -1.0, float("inf"), float("nan")):
        assert error_of(params(), capi.make_adaptive(t, 64)) == (inv, target), t
    floor = "lt_render_adaptive: floor must be finite and >= 0"
    for f in (-1e-6, float("inf"), float("nan")):
        assert error_of(params(), capi.make_adaptive(0.05, 64, floor=f)) == (inv, floor), f
    assert rounds(16, 64) == capi.adaptive_rounds(params(), capi.make_adaptive(0.05, 64, floor=0.5))
    assert error_of(params(), capi.make_adaptive(0.05, 64, round_frames=-1)) == (
        inv, "lt_render_adaptive: round_frames must be >= 0")
    assert error_of(params(), capi.make_adaptive(0.05, 15)) == (inv, "lt_render_adaptive: max_frames must be >= frames")
    assert error_of(params(), good, 0xFFFFFFF0) == (
        inv, "lt_render_adaptive: camera.frameCount + max_frames must fit 32 bits")
    bad_size = capi.make_adaptive(0.05, 64)
    bad_size.struct_size = 8
    assert error_of(params(), bad_size) == (inv, "lt_render_adaptive: aparams.struct_size mismatch")
    # the checks of lt_render come first, with their messages
    assert error_of(capi.make_params(L.KERNEL_GI, 0, H, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN), good) == (
        inv, "lt_render_adaptive: width/height must be > 0 and depth >= 3")
    assert error_of(capi.make_params(99, W, H, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN), good) == (
        uns, "lt_render_adaptive: unknown kernel id")
    # 2^31 pixels: the 32-bit pixel lists cannot number them
    big = capi.make_params(L.KERNEL_GI, 65536, 32768, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN)
    assert error_of(big, good) == (uns, "lt_render_adaptive: a masked call handles at most 2^31 - 1 pixels (width * height)")
    lib = capi.load()
    assert lib.lt_debug_adaptive_rounds(C.byref(params()), None, 0, None, 0) == inv
    assert lib.lt_last_error(None).decode() == "lt_render_adaptive: aparams is NULL"
    out = np.zeros(2, np.int32)
    assert lib.lt_debug_adaptive_rounds(C.byref(params()), C.byref(good), 0, out.ctypes.data, 2) == inv


@pytest.mark.parametrize("kernel", [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY, L.KERNEL_LIGHTING25,
                                    L.KERNEL_ACCUMULATOR, L.KERNEL_GI25, L.KERNEL_GI])
def test_every_kernel_id_is_accepted(kernel):
    p = capi.make_params(kernel, W, H, frames=4, accum_mode=L.ACCUM_RUNNING_MEAN)
    assert capi.adaptive_rounds(p, capi.make_adaptive(0.05, 16)) == [4, 4, 4, 4]


def test_null_context():
    lib = capi.load()
    p = params()
    a = capi.make_adaptive(0.05, 64)
    cam = L.make_camera(0, 2.5, -50)
    res = capi.AdaptiveResult()
    assert lib.lt_render_adaptive(None, None, cam.ctypes.data, C.byref(p), C.byref(a), None, None, C.byref(res)) == \
        capi.ERR_INVALID
    assert lib.lt_last_error(None).decode() == "lt_render_adaptive: ctx is NULL"
    assert lib.lt_render_adaptive_device(None, None, cam.ctypes.data, C.byref(p), C.byref(a), None, None, None,
                                         C.byref(res), 1) == capi.ERR_INVALID
    assert lib.lt_last_error(None).decode() == "lt_render_adaptive_device: ctx is NULL"
    assert lib.lt_debug_ctx_adaptive_part(None, 2, 0) == capi.ERR_INVALID
    assert lib.lt_last_error(None).decode() == "lt_debug_ctx_adaptive_part: ctx is NULL"


def test_scene_file_keys_reach_the_extension(tmp_path):
    scene = json.load(open("resources/scenes/cornell_global_illumination.scene"))
    path = str(tmp_path / "adaptive.scene")
    json.dump(scene, open(path, "w"))
    e = host.scene_extension(path)
    assert (e.adaptiveError, e.adaptiveRoundFrames, e.adaptiveMaxFrames) == (0.0, 0, 0)  # off unless asked for
    scene["renderer"].update({"frames": 16, "accumulate": True, "adaptive_error": 0.05, "adaptive_round_frames": 8,
                              "adaptive_max_frames": 48})
    json.dump(scene, open(path, "w"))
    e = host.scene_extension(path)
    assert (e.frames, e.accumulate) == (16, 1)
    assert (e.adaptiveError, e.adaptiveRoundFrames, e.adaptiveMaxFrames) == (np.float32(0.05), 8, 48)
    assert not e.pPixelFrames and e.adaptiveRounds == 0


@pytest.mark.parametrize("height", [1, 7, 8, 9, 75, 1080, 2160])
@pytest.mark.parametrize("devices", [1, 2, 3, 8])
def test_row_partition_covers_the_image_once(height, devices):
    """the rows each device of an adaptive call owns (the tile split's partition): every row exactly once, in whole
    blocks of 8 rows dealt round-robin"""
    rows = [capi.tile_rows(height, devices, g) for g in range(devices)]
    allrows = np.sort(np.concatenate(rows))
    assert (allrows == np.arange(height)).all()
    for g, r in enumerate(rows):
        assert ((r // 8) % devices == g).all()

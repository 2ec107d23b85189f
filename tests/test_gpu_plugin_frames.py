"""Plug-in kernels rendered like the built-in ones (lt_render_plugin_frames): many frames per call, combined into the
context's accumulator, divided among the devices of a multi-GPU context by the sample split; and the same through
RendererCUDA / RendererOpenCL with a RenderExtensionB200.

tests/plugins/gi_plugin.cu equals the built-in LT_KERNEL_GI frame for frame, and the fold kernel uses the built-in
pipelines' own FrameSink, so on one device the accumulated result must equal the built-in call bit for bit.  Across
devices the sample split sums per-device partial sums: bit-equal to the built-in kernel's sample split on the same
group, within 1e-5 relative of one GPU (the tolerance of test_gpu_multi.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L

PLUGINS = os.path.join(util.ROOT, "tests", "plugins")
GI = os.path.join(PLUGINS, "gi_plugin.cu")
ECHO = os.path.join(PLUGINS, "echo_buffers.cu")
BARY = os.path.join(PLUGINS, "cl_barycentric.cl")
LIGHT = os.path.join(PLUGINS, "cl_direct_light.cl")
GI_FILE = "examples/global_illumination/resources/kernels/global_illumination.cl"


def device_count():
    import torch
    return torch.cuda.device_count()


def rel_diff(a, b):
    return float((np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), 1e-3)).max())


def params(w, h, frames=1, accum=L.ACCUM_RUNNING_MEAN, stride=1, weight=0.0, block=(8, 8), **kw):
    p = capi.make_params(0, w, h, frames=frames, frame_stride=stride, accum_mode=accum, accum_weight=weight, **kw)
    p.block_x, p.block_y = block
    return p


def gi_params(w, h, **kw):
    """The built-in kernel gi_plugin.cu restates, 4 bounces"""
    return capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, **kw)


# ---------------------------------------------------------------- CPU: binding and arguments

def test_binding_and_null_context():
    lib = capi.load()
    assert hasattr(lib, "lt_render_plugin_frames")
    p = params(8, 8)
    cam = np.ascontiguousarray(util.default_camera(), dtype=L.CAMERA)
    out = np.full((8, 8, 3), 7.0, np.float32)
    rc = lib.lt_render_plugin_frames(None, None, cam.ctypes.data, 0, C.byref(p), 0, 0, out.ctypes.data)
    assert rc == capi.ERR_INVALID
    assert b"ctx is NULL" in lib.lt_last_error(None)
    assert (out == 7.0).all()


# ---------------------------------------------------------------- one GPU

@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens"])
def test_gi_plugin_frames_equal_the_builtin_kernel(ctx, name):
    pid = ctx.plugin_load(GI)
    sc = ctx.upload(util.scene(name))
    w, h = 320, 200
    for frames, stride, fc in ((1, 1, 0), (5, 1, 0), (3, 4, 2)):
        cam = util.default_camera(0.02, fc)
        ctx.accum_reset()
        got = ctx.render_plugin_frames(sc, cam, pid, params(w, h, frames, stride=stride))
        assert ctx.stats().kernel_launches == 2 * frames
        ctx.accum_reset()
        want = ctx.render(sc, cam, gi_params(w, h, frames=frames, frame_stride=stride, accum_mode=L.ACCUM_RUNNING_MEAN))
        util.assert_bit_equal(got, want, "%s: %d frames, stride %d, from frameCount %d" % (name, frames, stride, fc))
    # weighted sum on top of an accumulator that holds two frames (frameCount 0 discards what was there before)
    base, cam = util.default_camera(0.02, 0), util.default_camera(0.02, 6)
    ctx.render(sc, base, gi_params(w, h, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN))
    got = ctx.render_plugin_frames(sc, cam, pid, params(w, h, 4, accum=L.ACCUM_WEIGHTED_SUM, weight=0.25))
    ctx.render(sc, base, gi_params(w, h, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN))
    want = ctx.render(sc, cam, gi_params(w, h, frames=4, accum_mode=L.ACCUM_WEIGHTED_SUM, accum_weight=0.25))
    util.assert_bit_equal(got, want, "%s: weighted sum" % name)
    sc.release()


@pytest.mark.gpu
def test_gi_plugin_64_frames_at_1080p(ctx):
    """The benchmark workload (the built-in call runs the wavefront), its two-call continuation, and the cost of the
    frame loop against 64 single-frame calls."""
    pid = ctx.plugin_load(GI)
    sc = ctx.upload(util.scene("cornell_box"))
    w, h = 1920, 1080
    cam = util.default_camera(0.0, 0)
    got = ctx.render_plugin_frames(sc, cam, pid, params(w, h, 64))
    st = ctx.stats()
    assert st.kernel_launches == 128 and st.rays == 0 and st.node_tests == 0 and st.tri_tests == 0
    want = ctx.render(sc, cam, gi_params(w, h, frames=64, accum_mode=L.ACCUM_RUNNING_MEAN))
    util.assert_bit_equal(got, want, "64 frames at 1080p")
    # progressive: 32 + 32 frames, the second call continuing at frameCount 32
    ctx.render_plugin_frames(sc, cam, pid, params(w, h, 32), want_output=False)
    got2 = ctx.render_plugin_frames(sc, util.default_camera(0.0, 32), pid, params(w, h, 32))
    util.assert_bit_equal(got2, want, "32 + 32 frames")
    acc = np.empty_like(want)
    ctx.lib.lt_accum_read(ctx.h, acc.ctypes.data, acc.size)
    util.assert_bit_equal(acc, want, "lt_accum_read after a plug-in call")
    # kernel time of the call against 64 single-frame plug-in calls
    ctx.render_plugin_frames(sc, cam, pid, params(w, h, 64), want_output=False)
    frames_ms = ctx.stats().kernel_ms
    single_ms = 0.0
    for k in range(64):
        ctx.render_plugin(sc, util.default_camera(0.0, k), pid, w, h, block=(8, 8))
        single_ms += ctx.stats().kernel_ms
    print("64-frame call %.2f ms, 64 single-frame calls %.2f ms" % (frames_ms, single_ms))
    assert frames_ms <= 1.1 * single_ms, (frames_ms, single_ms)
    sc.release()


@pytest.mark.gpu
def test_gi_plugin_frames_on_a_large_mesh(ctx, tmp_path):
    """A tree too large for the threaded copies: the plug-in's stack traversal"""
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 200, 0x5EED)  # 80 012 triangles, 160 023 nodes
    sc = ctx.upload(host.load_scene_buffers(p))
    pid = ctx.plugin_load(GI)
    for frames, stride, fc in ((1, 1, 0), (5, 1, 0), (3, 4, 2)):
        cam = util.default_camera(0.0, fc)
        ctx.accum_reset()
        got = ctx.render_plugin_frames(sc, cam, pid, params(320, 200, frames, stride=stride))
        ctx.accum_reset()
        want = ctx.render(sc, cam, gi_params(320, 200, frames=frames, frame_stride=stride,
                                             accum_mode=L.ACCUM_RUNNING_MEAN))
        util.assert_bit_equal(got, want, "synthetic mesh: %d frames, stride %d" % (frames, stride))
    sc.release()


@pytest.mark.gpu
def test_frame_numbering(ctx):
    """echo_buffers.cu writes position.z + x + frameCount in channel 0: frame k of a call sees fc + k * stride"""
    pid = ctx.plugin_load(ECHO)
    sc = ctx.upload(util.scene("cornell_box"))
    w, h, F, fc, stride = 64, 40, 5, 7, 3
    singles = [ctx.render_plugin(sc, util.default_camera(0.0, fc + k * stride), pid, w, h, block=(8, 8))
               for k in range(F)]
    x = np.arange(w, dtype=np.float32)[None, :]
    for k, s in enumerate(singles):
        want0 = (np.float32(-50.0) + x) + np.float32(fc + k * stride)
        util.assert_bit_equal(s[..., 0], np.broadcast_to(want0, (h, w)), "frame %d" % k)
    ctx.accum_reset()
    got = ctx.render_plugin_frames(sc, util.default_camera(0.0, fc), pid,
                                   params(w, h, F, accum=L.ACCUM_WEIGHTED_SUM, stride=stride, weight=1.0))
    want = np.zeros_like(singles[0])
    for s in singles:
        want = want + s
    util.assert_bit_equal(got, want, "weighted sum of the frames")
    # LT_ACCUM_NONE: the frames go to the output in order, as F single-frame calls
    got = ctx.render_plugin_frames(sc, util.default_camera(0.0, fc), pid, params(w, h, F, accum=L.ACCUM_NONE, stride=stride))
    assert ctx.stats().kernel_launches == F
    util.assert_bit_equal(got, singles[-1], "LT_ACCUM_NONE")
    sc.release()


@pytest.mark.gpu
@pytest.mark.parametrize("path", [BARY, LIGHT])
@pytest.mark.parametrize("work_block,group", [((0, 0), (0, 0)), ((24, 16), (8, 4))])
def test_opencl_plugin_frames_equal_the_per_frame_protocol(ctx, path, work_block, group):
    """RUNNING_MEAN over 6 frames equals the host running mean (lt_oracle.accumulate) of 6 lt_render_plugin_cl frames"""
    pid = ctx.plugin_load(path)
    sc = ctx.upload(util.scene("cornell_box"))
    w, h = 101, 75
    want = np.zeros((h, w, 3), np.float32)
    for k in range(6):
        one = ctx.render_plugin_cl(sc, util.default_camera(0.0, k), pid, w, h, work_block=work_block, group=group)
        O.accumulate(want, one, k)
    got = ctx.render_plugin_frames(sc, util.default_camera(0.0, 0), pid, params(w, h, 6, block=group),
                                   work_block=work_block)
    util.assert_bit_equal(got, want, "%s, work block %s" % (os.path.basename(path), work_block))
    assert got.any()
    if work_block != (0, 0):
        cw, ch = w // work_block[0] * work_block[0], h // work_block[1] * work_block[1]
        assert not got[ch:].any() and not got[:, cw:].any(), "uncovered pixels stay 0"
        assert ctx.stats().kernel_launches == 6 * ((w // work_block[0]) * (h // work_block[1]) + 1)
    sc.release()


def call_raw(c, sc, pid, p, work_block=(0, 0), camera=None, scene_h=None):
    """lt_render_plugin_frames into a buffer of 7.0: (return code, whether the buffer is untouched)"""
    cam = np.ascontiguousarray(util.default_camera() if camera is None else camera, dtype=L.CAMERA)
    out = np.full((p.height, p.width, max(p.depth, 3)), 7.0, np.float32)
    rc = c.lib.lt_render_plugin_frames(c.h, sc.h if scene_h is None else scene_h, cam.ctypes.data, pid, C.byref(p),
                                       work_block[0], work_block[1], out.ctypes.data)
    return rc, bool((out == 7.0).all())


@pytest.mark.gpu
def test_argument_errors(ctx):
    gi = ctx.plugin_load(GI)
    cl = ctx.plugin_load(BARY)
    sc = ctx.upload(util.scene("cornell_box"))
    ok = params(32, 16, 2)
    assert call_raw(ctx, sc, gi, ok) == (0, False)
    for flag in (1 << 0, 1 << 7, 1 << 1):  # LT_FLAG_STATS, LT_FLAG_STATS_TRACED, LT_FLAG_CULL
        assert call_raw(ctx, sc, gi, params(32, 16, 2, flags=flag)) == (capi.ERR_UNSUPPORTED, True), flag
    # the schedule flags do not apply and are ignored
    assert call_raw(ctx, sc, gi, params(32, 16, 2, flags=(1 << 2) | (1 << 5)))[0] == 0
    for bad in (-1, 99):
        assert call_raw(ctx, sc, bad, ok) == (capi.ERR_INVALID, True)
    assert call_raw(ctx, sc, gi, ok, work_block=(16, 8)) == (capi.ERR_INVALID, True)  # work block: .cl only
    assert call_raw(ctx, sc, cl, ok, work_block=(-1, 0)) == (capi.ERR_INVALID, True)
    assert call_raw(ctx, sc, cl, params(32, 16, 2, block=(5, 5))) == (capi.ERR_INVALID, True)  # group must divide
    for field, value in (("struct_size", 12), ("width", 0), ("depth", 2), ("frames", 0), ("accum_mode", 3)):
        p = params(32, 16, 2)
        setattr(p, field, value)
        assert call_raw(ctx, sc, gi, p) == (capi.ERR_INVALID, True), field
    assert call_raw(ctx, sc, gi, ok, scene_h=0) == (capi.ERR_INVALID, True)
    # kernel and max_ray_depth are ignored
    p = params(32, 16, 2)
    p.kernel, p.max_ray_depth = 99, 999
    assert call_raw(ctx, sc, gi, p)[0] == 0
    # the single-frame entry points still refuse a plug-in of the other language
    with pytest.raises(capi.LtError, match="OpenCL C kernel"):
        ctx.render_plugin(sc, util.default_camera(), cl, 32, 16)
    with pytest.raises(capi.LtError, match="CUDA kernel"):
        ctx.render_plugin_cl(sc, util.default_camera(), gi, 32, 16)
    sc.release()


# ---------------------------------------------------------------- several GPUs

@pytest.mark.gpu
@pytest.mark.parametrize("exchange", ["nccl", "p2p"])
def test_sample_split_of_a_plugin(exchange, monkeypatch):
    util.skip_nccl_without_two_gpus(exchange)
    monkeypatch.setenv("LT_MULTI_EXCHANGE", exchange)
    for n in util.group_sizes():
        sample_split_of_a_plugin(exchange, n)


def sample_split_of_a_plugin(exchange, n):
    sb = util.scene("cornell_box")
    one, many = capi.Context(0), util.device_group(n)
    s1, sm = one.upload(sb), many.upload(sb)
    p1, pm = one.plugin_load(GI), many.plugin_load(GI)
    cam = util.default_camera(0.0, 0)
    for w, h, frames in ((640, 360, 16), (1920, 1080, 8)):
        want1 = one.render_plugin_frames(s1, cam, p1, params(w, h, frames))
        got = many.render_plugin_frames(sm, cam, pm, params(w, h, frames, split_mode=L.SPLIT_SAMPLES))
        builtin = many.render(sm, cam, gi_params(w, h, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                                                 split_mode=L.SPLIT_SAMPLES))
        util.assert_bit_equal(got, builtin, "%s %dx%d: plug-in vs built-in sample split" % (exchange, w, h))
        assert rel_diff(got, want1) <= 1e-5, (exchange, w, h, rel_diff(got, want1))
        # AUTO is the sample split; two calls continue the accumulator
        half = frames // 2
        many.render_plugin_frames(sm, cam, pm, params(w, h, half), want_output=False)
        got2 = many.render_plugin_frames(sm, util.default_camera(0.0, half), pm, params(w, h, frames - half))
        assert rel_diff(got2, want1) <= 1e-5
    # an OpenCL C plug-in on the group
    c1, cm = one.plugin_load(LIGHT), many.plugin_load(LIGHT)
    want = one.render_plugin_frames(s1, cam, c1, params(101, 75, 6, block=(0, 0)))
    got = many.render_plugin_frames(sm, cam, cm, params(101, 75, 6, block=(0, 0)))
    assert got.any() and rel_diff(got, want) <= 1e-5
    # what a group refuses, leaving the buffer untouched
    assert call_raw(many, sm, pm, params(64, 48, 4, split_mode=L.SPLIT_TILES)) == (capi.ERR_UNSUPPORTED, True)
    assert call_raw(many, sm, pm, params(64, 48, 4, accum=L.ACCUM_NONE)) == (capi.ERR_UNSUPPORTED, True)
    assert call_raw(many, sm, pm, params(64, 48, 4, stride=2)) == (capi.ERR_UNSUPPORTED, True)
    assert call_raw(many, sm, 99, params(64, 48, 4)) == (capi.ERR_INVALID, True)
    with pytest.raises(capi.LtError, match="single-GPU"):
        many.render_plugin(sm, cam, pm, 64, 48)
    sm.release(); many.close(); s1.release(); one.close()


# ---------------------------------------------------------------- the C++ surface

@pytest.fixture
def world():
    os.chdir(util.ROOT)  # resource paths are CWD-relative
    cam = host.Camera(0, 2.5, -50, 0)
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model)
    yield cam, model, accel
    accel.close(); model.close(); cam.close()


@pytest.mark.gpu
def test_renderer_cuda_honours_the_extension_for_a_plugin(world):
    cam, model, accel = world
    r = host.Renderer(host.PLATFORM_CUDA)
    w, h = 320, 200
    ext = host.make_extension(frames=8, accumulate=True, max_ray_depth=4)
    want = r.render(GI_FILE, w, h, accel, model, cam, block=(8, 8), ext=ext)
    got = r.render("tests/plugins/gi_plugin.cu", w, h, accel, model, cam, block=(8, 8), ext=ext)
    util.assert_bit_equal(got, want, "RendererCUDA: gi_plugin.cu vs the built-in GI file, 8 frames")
    assert ext.kernelMilliseconds > 0 and ext.rays == 0
    if device_count() >= 2:
        ext2 = host.make_extension(frames=8, accumulate=True, max_ray_depth=4, devices=2)
        got2 = r.render("tests/plugins/gi_plugin.cu", w, h, accel, model, cam, block=(8, 8), ext=ext2)
        assert rel_diff(got2, want) <= 1e-5
    r.close()


@pytest.mark.gpu
def test_renderer_opencl_honours_the_extension_for_a_plugin(world):
    cam, model, accel = world
    r = host.Renderer(host.PLATFORM_OPENCL)
    w, h = 101, 75
    path = "tests/plugins/cl_direct_light.cl"
    want = np.zeros((h, w, 3), np.float32)
    for k in range(6):
        cam.set_frame_count(k)
        O.accumulate(want, r.render(path, w, h, accel, model, cam), k)
    cam.set_frame_count(0)
    got = r.render(path, w, h, accel, model, cam, ext=host.make_extension(frames=6, accumulate=True))
    util.assert_bit_equal(got, want, "RendererOpenCL: 6 accumulated frames vs the per-frame protocol")
    r.close()


@pytest.mark.gpu
def test_multi_gpu_example_with_a_user_kernel():
    subprocess.check_call(["make", "-C", os.path.join(util.ROOT, "examples"), "-s"])
    n = max(1, min(device_count(), 8))
    r = subprocess.run([os.path.join(util.ROOT, "examples", "bin", "multi_gpu"), "--devices", str(n), "--size", "320",
                        "200", "--frames", "8", "--kernel", "tests/plugins/cl_direct_light.cl"], cwd=util.ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "cl_direct_light.cl" in r.stdout and "GPUs:" in r.stdout

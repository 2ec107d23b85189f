"""The plug-in device API from OpenCL C: a .cl file that includes lens_trace_b200_device_cl.h calls the library's own
traversal, RNG and sampling (lt_trace, lt_occluded, lt_random, lt_sample_light, lt_sample_hemisphere, ...).

tests/plugins/gi_plugin.cl is the example's global-illumination kernel ported to that API.  It computes what the
built-in LT_KERNEL_GI pipeline computes, in the same operation order, so on one device the two must agree bit for bit,
whatever the work block and work-group of the launch."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import util
from lens_trace_b200 import capi, host, layouts as L

PLUGINS = os.path.join(util.ROOT, "tests", "plugins")
GI_CL = os.path.join(PLUGINS, "gi_plugin.cl")
GI_CU = os.path.join(PLUGINS, "gi_plugin.cu")
LIGHT = os.path.join(PLUGINS, "cl_direct_light.cl")
GI_FILE = "examples/global_illumination/resources/kernels/global_illumination.cl"
INCLUDE = '#include "lens_trace_b200_device_cl.h"\n'
SIG = ("__global float* nodes, __global float* primitives, __global float* materials, __global float* lights, "
       "__global float* camera, __global float* output, uint currentBlock, uint width, uint height, uint depth")
TRACE_CALL = ("  LtHit h = lt_trace((float4)(0.0f, 0.0f, 0.0f, 1.0f), (float4)(0.0f, 0.0f, 1.0f, 0.0f), FLT_MAX, -1, 0, "
              "LT_EPSILON_GI);\n  output[0] = h.t;\n")


def _compile_text(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return capi.compile_cl(str(p))


# ---------------------------------------------------------------- CPU tests

def test_the_ported_gi_kernel_compiles():
    ok, log = capi.compile_cl(GI_CL)
    assert ok, log


def test_the_include_line_becomes_an_empty_line():
    src = "// a kernel\n" + INCLUDE + "  #  include   \"lens_trace_b200_device_cl.h\"\nint a;\n"
    got, off = capi.translate_cl(src)
    assert not off
    assert got.split("\n") == ["// a kernel", "", "  ", "int a;", ""]
    # any other include stays for NVRTC to resolve
    other = '#include "my_helpers.h"\n'
    assert capi.translate_cl(other)[0] == other


def test_an_error_after_the_include_names_its_own_line(tmp_path):
    ok, log = _compile_text(tmp_path, "typo.cl", "// a kernel\n" + INCLUDE + "\n__kernel void linearKernel(%s) {\n"
                            "%s  output[1] = 1.0f\n}\n" % (SIG, TRACE_CALL))
    assert not ok
    assert re.search(r"typo\.cl\(8\): error", log), log  # the missing ';' is seen at the '}' of line 8
    ok, log = _compile_text(tmp_path, "fine.cl", "// a kernel\n" + INCLUDE + "\n__kernel void linearKernel(%s) {\n"
                            "%s}\n" % (SIG, TRACE_CALL))
    assert ok, log


def test_calling_the_api_without_the_include_fails_at_the_users_line(tmp_path):
    ok, log = _compile_text(tmp_path, "noinc.cl", "// a kernel\n\n__kernel void linearKernel(%s) {\n%s}\n"
                            % (SIG, TRACE_CALL))
    assert not ok
    assert re.search(r"noinc\.cl\(4\): error", log), log
    assert "lt_trace" in log or "LtHit" in log, log


def test_the_reference_names_live_next_to_the_api(tmp_path):
    """cl_direct_light.cl defines the reference's own Ray, Payload, random, intersect and cameraRay; with the include
    added it still compiles, and it can call the API next to its own functions."""
    text = open(LIGHT).read()
    for name in ("typedef struct Ray", "typedef struct Payload", "float random(", "void intersect(", "Ray cameraRay("):
        assert name in text
    ok, log = _compile_text(tmp_path, "cl_direct_light.cl", INCLUDE + text)
    assert ok, log
    store = "  output[id + 0] = colour.x;"
    assert store in text
    mixed = text.replace(store, "  output[id + 0] = colour.x + (float)lt_is_light(payload.primitiveIndex) * "
                                "lt_random(film, 1.0f) + (float)lt_occluded(ray.origin, ray.direction, 1.0f, -1, "
                                "LT_EPSILON_BASIC);")
    ok, log = _compile_text(tmp_path, "mixed.cl", INCLUDE + mixed)
    assert ok, log


def test_including_the_cuda_header_names_the_opencl_one(tmp_path):
    ok, log = _compile_text(tmp_path, "wrong.cl", "// a kernel\n#include \"lens_trace_b200_device.cuh\"\n"
                            "__kernel void linearKernel(%s) {\n%s}\n" % (SIG, TRACE_CALL))
    assert not ok
    assert re.search(r"wrong\.cl\(2\)", log), log
    assert "lens_trace_b200_device_cl.h" in log, log


# ---------------------------------------------------------------- GPU tests

@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def gi_params(w, h, kernel_mode=0, **kw):
    """The built-in kernel gi_plugin.cl restates, 4 bounces"""
    return capi.make_params(L.KERNEL_GI, w, h, kernel_mode=kernel_mode, max_ray_depth=4, **kw)


def frame_params(w, h, frames, group=(0, 0), split_mode=0):
    p = capi.make_params(0, w, h, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN, split_mode=split_mode)
    p.block_x, p.block_y = group
    return p


def stack_depth(c, sc):
    sd = C.c_int32()
    assert c.lib.lt_scene_info(sc.h, None, None, C.byref(sd)) == 0
    return sd.value


def traversal_smem(levels, threads):
    """Dynamic shared memory lt_trace needs per block: (stack levels + 16 leaf-FIFO entries) ints per thread"""
    return (levels + 16) * 4 * threads


# (work block, group): MAX_FIT with the library's group, an 8x8 group, and 160x100 work blocks (several launches)
SHAPES = [((0, 0), (0, 0)), ((0, 0), (8, 8)), ((160, 100), (0, 0))]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens"])
def test_gi_plugin_cl_equals_the_builtin_kernel(ctx, name, mode):
    pid = ctx.plugin_load(GI_CL)
    sc = ctx.upload(util.scene(name))
    w, h = 320, 200
    for frame in (0, 1, 9):
        cam = util.default_camera(0.02, frame)
        want = ctx.render(sc, cam, gi_params(w, h, mode))
        for wb, group in SHAPES:
            got = ctx.render_plugin_cl(sc, cam, pid, w, h, kernel_mode=mode, work_block=wb, group=group)
            util.assert_bit_equal(got, want, "%s frame %d mode %d work block %s group %s" % (name, frame, mode, wb, group))
            if wb != (0, 0):
                assert ctx.stats().kernel_launches == (w // wb[0]) * (h // wb[1])
    if mode == 0:
        assert want.max() <= 1.0
    sc.release()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_gi_plugin_cl_on_a_large_mesh(ctx, tmp_path, mode):
    """A tree too large for the threaded copies: lt_trace walks the stack traversal in the launch's dynamic shared
    memory; one group needs more than the 48 KB a launch gets without asking."""
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 200, 0x5EED)  # 80 012 triangles, 160 023 nodes
    sc = ctx.upload(host.load_scene_buffers(p))
    pid = ctx.plugin_load(GI_CL)
    w, h = 400, 240
    big = (40, 12)
    smem = traversal_smem(stack_depth(ctx, sc), big[0] * big[1])
    assert 48 * 1024 < smem <= 200 * 1024, smem
    cam = util.default_camera(0.0, 2)
    want = ctx.render(sc, cam, gi_params(w, h, mode))
    for wb, group in [((0, 0), (0, 0)), ((0, 0), (8, 8)), ((200, 120), (8, 8)), ((0, 0), big)]:
        got = ctx.render_plugin_cl(sc, cam, pid, w, h, kernel_mode=mode, work_block=wb, group=group)
        util.assert_bit_equal(got, want, "synthetic mesh mode %d work block %s group %s" % (mode, wb, group))
    sc.release()


@pytest.mark.gpu
def test_gi_plugin_cl_64_frames_at_1080p(ctx):
    pid = ctx.plugin_load(GI_CL)
    sc = ctx.upload(util.scene("cornell_box"))
    w, h = 1920, 1080
    cam = util.default_camera(0.0, 0)
    got = ctx.render_plugin_frames(sc, cam, pid, frame_params(w, h, 64))
    want = ctx.render(sc, cam, gi_params(w, h, frames=64, accum_mode=L.ACCUM_RUNNING_MEAN))
    util.assert_bit_equal(got, want, "64 frames at 1080p")
    # progressive: 32 + 32 frames, the second call continuing at frameCount 32
    ctx.render_plugin_frames(sc, cam, pid, frame_params(w, h, 32), want_output=False)
    got2 = ctx.render_plugin_frames(sc, util.default_camera(0.0, 32), pid, frame_params(w, h, 32))
    util.assert_bit_equal(got2, want, "32 + 32 frames")
    sc.release()


@pytest.mark.gpu
def test_renderer_opencl_renders_the_ported_file_with_an_extension():
    os.chdir(util.ROOT)  # resource paths are CWD-relative
    cam = host.Camera(0, 2.5, -50, 0)
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model)
    r = host.Renderer(host.PLATFORM_OPENCL)
    w, h = 320, 200
    ext = host.make_extension(frames=8, accumulate=True, max_ray_depth=4)
    want = r.render(GI_FILE, w, h, accel, model, cam, ext=ext)
    got = r.render("tests/plugins/gi_plugin.cl", w, h, accel, model, cam, ext=ext)
    util.assert_bit_equal(got, want, "RendererOpenCL: gi_plugin.cl vs the built-in GI file, 8 frames")
    assert got.any()
    r.close(); accel.close(); model.close(); cam.close()


def comb_scene(depth):
    """A tree of `depth` inner nodes in a chain (each one's second child a leaf): its traversal stack needs `depth`
    levels.  Every node has the box of the whole scene."""
    n = 2 * depth + 1
    nodes = np.zeros(n, L.NODE)
    prims = np.zeros(depth + 1, L.PRIM)
    for k in range(depth + 1):
        x = float(k)
        prims["a"][k], prims["b"][k], prims["c"][k] = (x, 0, 10), (x + 1, 0, 10), (x, 1, 10)
        for c in ("na", "nb", "nc"):
            prims[c][k] = (0, 0, -1)
    nodes["min"] = (0, 0, 10)
    nodes["max"] = (depth + 1, 1, 10)
    for k in range(depth):
        nodes["offset"][k] = 2 * depth - k  # second child: a leaf after the chain
        nodes["offset"][2 * depth - k] = k + 1
        nodes["count"][2 * depth - k] = 1
    nodes["offset"][depth], nodes["count"][depth] = 0, 1
    mats = np.zeros(1, L.MATERIAL)
    mats["diffuse"][0] = (0.5, 0.5, 0.5)
    return L.SceneBuffers(nodes, prims, mats, np.zeros(1, L.LIGHTS))


@pytest.mark.gpu
def test_a_group_whose_stacks_do_not_fit_is_refused():
    c = capi.Context(0)
    c.debug_limits(0, 100000)  # no host-built threaded copies: lt_trace walks the stack traversal
    sc = c.upload(comb_scene(40))
    levels = stack_depth(c, sc)
    assert levels == 40
    pid = c.plugin_load(GI_CL)
    w, h, group = 64, 64, (32, 32)
    assert traversal_smem(levels, group[0] * group[1]) > 200 * 1024
    cam = np.ascontiguousarray(util.default_camera(), dtype=L.CAMERA)
    out = np.full((h, w, 3), 7.0, np.float32)
    rc = c.lib.lt_render_plugin_cl(c.h, sc.h, cam.ctypes.data, pid, 0, w, h, 3, 0, 0, group[0], group[1],
                                   out.ctypes.data)
    assert rc == capi.ERR_INVALID and (out == 7.0).all()
    assert b"too large" in c.lib.lt_last_error(c.h)
    rc = c.lib.lt_render_plugin_frames(c.h, sc.h, cam.ctypes.data, pid, C.byref(frame_params(w, h, 4, group)), 0, 0,
                                       out.ctypes.data)
    assert rc == capi.ERR_INVALID and (out == 7.0).all()
    # a group that fits renders on the same scene
    small = (16, 16)
    assert 48 * 1024 < traversal_smem(levels, small[0] * small[1]) <= 200 * 1024
    c.render_plugin_cl(sc, util.default_camera(), pid, w, h, group=small)
    sc.release()
    c.close()


def rel_diff(a, b):
    return float((np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), 1e-3)).max())


@pytest.mark.gpu
def test_sample_split_of_the_ported_file():
    for n in util.group_sizes():
        sample_split_of_the_ported_file(n)


def sample_split_of_the_ported_file(n):
    sb = util.scene("cornell_box")
    one, many = capi.Context(0), util.device_group(n)
    s1, sm = one.upload(sb), many.upload(sb)
    p1, pm = one.plugin_load(GI_CL), many.plugin_load(GI_CL)
    cam = util.default_camera(0.0, 0)
    for w, h, frames in ((640, 360, 16), (1920, 1080, 8)):
        want1 = one.render_plugin_frames(s1, cam, p1, frame_params(w, h, frames))
        got = many.render_plugin_frames(sm, cam, pm, frame_params(w, h, frames, split_mode=L.SPLIT_SAMPLES))
        builtin = many.render(sm, cam, gi_params(w, h, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                                                 split_mode=L.SPLIT_SAMPLES))
        util.assert_bit_equal(got, builtin, "%dx%d: gi_plugin.cl vs built-in sample split" % (w, h))
        assert rel_diff(got, want1) <= 1e-5, (w, h, rel_diff(got, want1))
    sm.release(); many.close(); s1.release(); one.close()


@pytest.mark.gpu
def test_gi_plugin_cl_kernel_time(ctx):
    """One 1080p frame on the Cornell box: within 1.5x of the built-in single-frame launch (the bound the .cu port
    keeps)."""
    pid = ctx.plugin_load(GI_CL)
    sc = ctx.upload(util.scene("cornell_box"))
    cam = util.default_camera(0.0, 3)
    t_plugin, t_builtin = [], []
    for _ in range(5):
        ctx.render_plugin_cl(sc, cam, pid, 1920, 1080)
        t_plugin.append(ctx.stats().kernel_ms)
        ctx.render(sc, cam, gi_params(1920, 1080), want_output=False)
        t_builtin.append(ctx.stats().kernel_ms)
    print("gi_plugin.cl %.3f ms, built-in %.3f ms" % (min(t_plugin), min(t_builtin)))
    assert min(t_plugin) <= 1.5 * min(t_builtin), (min(t_plugin), min(t_builtin))
    sc.release()

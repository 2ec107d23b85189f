"""User-written OpenCL C kernel files (.cl) compiled by NVRTC for sm_100a and launched like the reference's OpenCL
backend launches them (lt_plugin_load / lt_render_plugin_cl, RendererOpenCL::render).

The kernels under tests/plugins/*.cl are written in the reference's style (32-byte node stack traversal,
Moller-Trumbore, the 10-argument entry points).  The oracle is the same text run on the CPU: tests/cl_host/
cl_file_host.cpp compiles one file through oracle/cl_shim with g++, with the same vector-literal rewrite and the
same launch loop as oracle/cl_shim/ref_cl_host.cpp."""
import ctypes as C
import glob
import json
import os
import re
import subprocess
import time

import numpy as np
import pytest

import util
from lens_trace_b200 import capi, host, layouts as L

PLUGINS = os.path.join(util.ROOT, "tests", "plugins")
BARY = os.path.join(PLUGINS, "cl_barycentric.cl")
LIGHT = os.path.join(PLUGINS, "cl_direct_light.cl")
TILE = os.path.join(PLUGINS, "cl_tile_groups.cl")
SIG = ("__global float* nodes, __global float* primitives, __global float* materials, __global float* lights, "
       "__global float* camera, __global float* output, uint currentBlock, uint width, uint height, uint depth")
CASES = [("cornell_box", 128, 96), ("cornell_box_lens", 128, 96), ("cornell_box", 101, 75)]


# ---------------------------------------------------------------- CPU oracle: the same text through oracle/cl_shim

_oracles = {}


def cpu_oracle(path, workdir):
    """ctypes handle of `path` compiled for the CPU through oracle/cl_shim (cached per path)."""
    if path in _oracles:
        return _oracles[path]
    text = open(path).read()
    name = os.path.splitext(os.path.basename(path))[0]
    inc = os.path.join(workdir, name + ".inc")
    with open(inc, "w") as f:
        f.write(re.sub(r"\((float[234])\)\(", r"\1(", text))  # oracle/build_ref_cl.sh's rewrite
    so = os.path.join(workdir, "lib%s.so" % name)
    defs = ["-DLT_CL_FILE=\"%s\"" % inc]
    if re.search(r"__kernel\s+void\s+linearKernel\b", text):
        defs.append("-DLT_CL_LINEAR")
    if re.search(r"__kernel\s+void\s+tileKernel\b", text):
        defs.append("-DLT_CL_TILE")
    # oracle/build_ref_cl.sh's flags: one rounding per operation, nothing contracted
    subprocess.check_call(["g++", "-std=gnu++20", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-w",
                           "-Wno-narrowing", "-I", os.path.join(util.ROOT, "oracle", "cl_shim")] + defs +
                          [os.path.join(util.ROOT, "tests", "cl_host", "cl_file_host.cpp"), "-o", so, "-lpthread"])
    lib = C.CDLL(so)
    lib.clfile_render.argtypes = [C.c_int] + [C.c_void_p] * 6 + [C.c_int] * 8
    _oracles[path] = lib
    return lib


def cpu_render(lib, sb, cam, w, h, mode=0, work_block=(0, 0), group=(1, 1), depth=3):
    wb = (work_block[0] or w, work_block[1] or h)
    out = np.zeros((h, w, depth), np.float32)  # pixels outside every work block: 0, as lt_render_plugin_cl writes
    cam = np.ascontiguousarray(cam, dtype=L.CAMERA)
    rc = lib.clfile_render(mode, sb.nodes.ctypes.data, sb.prims.ctypes.data, sb.materials.ctypes.data,
                           sb.lights.ctypes.data, cam.ctypes.data, out.ctypes.data, w, h, depth, wb[0], wb[1], group[0],
                           group[1], 0)
    assert rc == 0
    return out


@pytest.fixture(scope="module")
def oracle_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("cl_oracle"))


# ---------------------------------------------------------------- CPU tests

@pytest.mark.parametrize("t", ["float", "int", "uint"])
@pytest.mark.parametrize("n", [2, 3, 4])
def test_vector_literal_rewrite_every_type(t, n):
    v = "%s%d" % (t, n)
    args = ", ".join(["1"] * n)
    src = "x = (%s)(%s); y = ( %s )\t(%s); z = (%s)s; w = f((%s)(%s));" % (v, args, v, args, v, v, args)
    got, off = capi.translate_cl(src)
    assert got == "x = %s(%s); y = %s(%s); z = (%s)s; w = f(%s(%s));" % (v, args, v, args, v, v, args)
    assert not off


def test_vector_literal_rewrite_nested_and_in_context():
    src = ("float4 a = (float4)((float3)((float2)(0.5f, (float)(1)), 2.0f), (a.x + (b.y * (c))));\n"
           "#define WHITE (float4)(1.0f, 1.0f, 1.0f, 1.0f)\n"
           "// (float4)(in a comment) stays\n"
           "/* (int2)(in a block\n comment) stays */ s = \"(uint3)(in a string)\";\n"
           "q = (float4) ( (float) (x) );\n"
           "r = (myfloat4)(x); p = (float5)(y);\n")
    got, _ = capi.translate_cl(src)
    assert got == ("float4 a = float4(float3(float2(0.5f, (float)(1)), 2.0f), (a.x + (b.y * (c))));\n"
                   "#define WHITE float4(1.0f, 1.0f, 1.0f, 1.0f)\n"
                   "// (float4)(in a comment) stays\n"
                   "/* (int2)(in a block\n comment) stays */ s = \"(uint3)(in a string)\";\n"
                   "q = float4( (float) (x) );\n"
                   "r = (myfloat4)(x); p = (float5)(y);\n")


def test_translation_keeps_lines_constant_data_and_pragmas():
    src = ("#pragma OPENCL EXTENSION cl_khr_fp64 : enable\n"
           "__constant float K[2] = {1.0f, 2.0f};\n"
           "constant int N = 3;\n"
           "float f(__constant float* k, constant int* n) { return k[0]; }\n"
           "__kernel void linearKernel() { __constant float* p = K; }\n")
    got, off = capi.translate_cl(src)
    assert not off
    lines = got.split("\n")
    assert len(lines) == len(src.split("\n"))  # every line stays where it was: messages point at the user's lines
    assert lines[0].strip() == ""
    assert lines[1] == "__constant__ const float K[2] = {1.0f, 2.0f};"
    assert lines[2] == "__constant__ const int N = 3;"
    assert lines[3] == "float f(const float* k, const int* n) { return k[0]; }"
    assert lines[4] == "__device__ void linearKernel() { const float* p = K; }"
    got, _ = capi.translate_cl("kernel void tileKernel(global float* a, __global const float* b, private int c) {}")
    assert got == "__device__ void tileKernel( float* a,  const float* b,  int c) {}"
    _, off = capi.translate_cl("// x\n  #  pragma   OPENCL FP_CONTRACT OFF\nint a;\n")
    assert off
    _, off = capi.translate_cl("#pragma OPENCL FP_CONTRACT ON\n// #pragma OPENCL FP_CONTRACT OFF\n")
    assert not off


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(PLUGINS, "*.cl"))), ids=os.path.basename)
def test_every_test_kernel_compiles_for_sm100a(path):
    t = time.perf_counter()
    ok, log = capi.compile_cl(path)
    dt = time.perf_counter() - t
    assert ok, log
    print("%s: translation + NVRTC compile for sm_100a %.1f ms" % (os.path.basename(path), dt * 1e3))


def _compile_text(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return capi.compile_cl(str(p))


def test_syntax_error_names_file_and_line(tmp_path):
    ok, log = _compile_text(tmp_path, "typo.cl", "// a kernel\n__kernel void linearKernel(%s) {\n  output[0] = 1.0f\n}\n"
                            % SIG)
    assert not ok
    assert re.search(r"typo\.cl\(4\): error", log), log  # the missing ';' is seen at the '}' of line 4


@pytest.mark.parametrize("body,what", [
    ("__local float tmp[16];\n  output[0] = tmp[0];", "lt_opencl_local_memory_is_not_supported"),
    ("barrier(0);", "barrier"),
    ("atomic_add((__global int*)output, 1);", "atomic_add"),
    ("half h = 1;", "lt_opencl_half_is_not_supported"),
    ("float4 v = (float4)(1.0f);\n  v = v * 2.0;\n  output[0] = v.x;", "double scalar"),
])
def test_unsupported_construct_is_an_error_at_the_users_line(tmp_path, body, what):
    ok, log = _compile_text(tmp_path, "unsupported.cl", "__kernel void linearKernel(%s) {\n  %s\n}\n" % (SIG, body))
    assert not ok
    assert what in log, log
    assert re.search(r"unsupported\.cl\(\d+\)|line \d+ of .*unsupported\.cl", log), log


@pytest.mark.parametrize("decl", ["__kernel void linearKernel() {}",
                                  "__kernel void linearKernel(__global float* nodes, float x) {}",
                                  "__kernel void linearKernel(%s, int extra) {}" % SIG,
                                  "__kernel void linearKernel(uint a, %s) {}" % SIG[:SIG.rindex(",")]])
def test_a_linear_kernel_that_does_not_take_the_reference_arguments_is_rejected(tmp_path, decl):
    ok, log = _compile_text(tmp_path, "sig.cl", "// user kernel\n\n" + decl + "\n")
    assert not ok
    assert "sig.cl(3)" in log, log  # reported at the user's declaration


def test_a_file_without_entry_points_is_rejected(tmp_path):
    ok, log = _compile_text(tmp_path, "none.cl", "__kernel void shade(%s) {}\n" % SIG)
    assert not ok and "neither" in log


SIZES = ("typedef char float3_is_16_bytes[sizeof(float3) == 16 ? 1 : -1];\n"
         "typedef char float4_is_16_bytes[sizeof(float4) == 16 ? 1 : -1];\n"
         "typedef char int3_is_16_bytes[sizeof(int3) == 16 ? 1 : -1];\n"
         "typedef struct { float a; float3 b; } S;\n"
         "typedef char float3_aligned_16[sizeof(S) == 32 ? 1 : -1];\n")


def test_three_component_vectors_are_16_bytes(tmp_path):
    ok, log = _compile_text(tmp_path, "sizes.cl", SIZES + "__kernel void linearKernel(%s) {\n"
                            "  output[0] = sizeof(float3); output[1] = sizeof(float4); output[2] = sizeof(uint3);\n}\n"
                            % SIG)
    assert ok, log
    ok, log = _compile_text(tmp_path, "sizes12.cl", "typedef char no[sizeof(float3) == 12 ? 1 : -1];\n"
                            "__kernel void linearKernel(%s) {}\n" % SIG)
    assert not ok and "sizes12.cl(1)" in log


def test_the_subset_compiles(tmp_path):
    """Every part of the documented subset in one file (address spaces, vector types and swizzles, math, geometric
    and work-item built-ins, file-scope constant data)."""
    ok, log = _compile_text(tmp_path, "subset.cl", r"""
#pragma OPENCL EXTENSION cl_khr_fp64 : enable
__constant float K[2] = {1.0f, 2.0f};
constant float4 C4 = (float4)(1.0f, 2.0f, 3.0f, 4.0f);
float helper(__constant float* k, __private float x) { return k[1] * x; }
kernel void linearKernel(global float* n, global float* p, global float* m, global float* l, global float* c,
                         global float* output, uint b, uint w, uint h, uint d) {
  uint4 u = (uint4)(1u) + 2u;
  int3 i3 = (int3)(1, 2, 3) * 2 - (int3)(1);
  float3 f = (float3)((float2)(1.0f, 2.0f), 3.0f);
  float4 g = (float4)(f, 1);
  g.xyz = f * 2.0f;
  g.xy = (float2)(0.5f);
  g += 1.0f; g *= 2; g /= (float4)(3.0f); g -= C4;
  float s = helper(K, dot(f, f)) + length(g) + distance(g, C4) + dot(normalize(g), cross(g, C4));
  s += clamp(0.5f, 0.0f, 1.0f) + min(1, 2) + max(1.0, 2.0) + pow(2.0f, 3.0f) + exp(1.0) + log(2.0f) + ceil(1.5f);
  s += fmin(f, 1.0f).x + fmax(f, f).y + clamp(f, 0.0f, 1.0f).z + fabs(-g).w + floor(g).x + sqrt(f).y;
  s += (float)u.w + (float)i3.z + fmod(5.0f, 3.0f) + sqrt(2.0) * cos(1.0) + sin(1.0f) + cross(f, f).x;
  s += get_global_id(0) + get_global_size(1) + get_local_id(2) + get_local_size(0) + get_group_id(1) + get_num_groups(2);
  output[0] = s;
}
""")
    assert ok, log


def test_cl_shim_runs_the_test_kernels(oracle_dir):
    """The CPU oracle itself: the test kernels run through oracle/cl_shim and draw what they say."""
    sb = util.scene("cornell_box")
    cam = util.default_camera()
    bary = cpu_render(cpu_oracle(BARY, oracle_dir), sb, cam, 64, 48)
    hit = bary.any(axis=-1)
    assert 0.2 < hit.mean() < 1.0
    np.testing.assert_allclose(bary[hit].sum(axis=-1), 1.0, atol=1e-5)
    assert (bary >= -1e-6).all() and (bary <= 1 + 1e-6).all()
    tile = cpu_render(cpu_oracle(TILE, oracle_dir), sb, cam, 64, 48, mode=1, work_block=(32, 16), group=(8, 4))
    want_x = ((np.arange(64) % 8) + 0.5) / 8
    want_y = ((np.arange(48) % 4) + 0.5) / 4
    np.testing.assert_array_equal(tile[..., 1], np.broadcast_to(want_x.astype(np.float32), (48, 64)))
    np.testing.assert_array_equal(tile[..., 2], np.broadcast_to(want_y.astype(np.float32)[:, None], (48, 64)))
    light = cpu_render(cpu_oracle(LIGHT, oracle_dir), sb, cam, 64, 48)
    assert light.max() > 0.1 and (light >= 0).all()
    # the reference's work blocks: a 24x20 block tiles 48x40 of 64x48, the rest stays 0
    part = cpu_render(cpu_oracle(BARY, oracle_dir), sb, cam, 64, 48, work_block=(24, 20), group=(8, 4))
    util.assert_bit_equal(part[:40, :48], bary[:40, :48])
    assert not part[40:].any() and not part[:, 48:].any()


# ---------------------------------------------------------------- GPU tests

@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def frac_within(got, want):
    return float(np.isclose(got, want, rtol=1e-4, atol=1e-6).all(axis=-1).mean())


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h", CASES)
@pytest.mark.parametrize("mode", [0, 1])
def test_barycentric_kernel_bit_for_bit(ctx, oracle_dir, name, w, h, mode):
    sb = util.scene(name)
    sc = ctx.upload(sb)
    pid = ctx.plugin_load(BARY)
    lib = cpu_oracle(BARY, oracle_dir)
    cam = util.default_camera()
    # MAX_FIT: one work block of the whole image, library's group
    got = ctx.render_plugin_cl(sc, cam, pid, w, h, kernel_mode=mode)
    want = cpu_render(lib, sb, cam, w, h, mode=mode)
    assert want.any()
    util.assert_bit_equal(got, want, "%s %dx%d mode %d MAX_FIT" % (name, w, h, mode))
    # a custom work block that leaves a remainder in both directions
    wb, grp = (24, 16), (8, 4)
    got = ctx.render_plugin_cl(sc, cam, pid, w, h, kernel_mode=mode, work_block=wb, group=grp)
    want = cpu_render(lib, sb, cam, w, h, mode=mode, work_block=wb, group=grp)
    util.assert_bit_equal(got, want, "%s %dx%d mode %d work block %s" % (name, w, h, mode, wb))
    cw, ch = w // wb[0] * wb[0], h // wb[1] * wb[1]
    assert (cw, ch) != (w, h)
    assert not got[ch:].any() and not got[:, cw:].any(), "remainder pixels are 0"
    assert ctx.stats().kernel_launches == (w // wb[0]) * (h // wb[1])
    sc.release()


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h", CASES)
def test_direct_light_kernel_close_to_cpu(ctx, oracle_dir, name, w, h):
    sb = util.scene(name)
    sc = ctx.upload(sb)
    pid = ctx.plugin_load(LIGHT)
    lib = cpu_oracle(LIGHT, oracle_dir)
    for frame in (0, 7):
        cam = util.default_camera(0.0, frame)
        got = ctx.render_plugin_cl(sc, cam, pid, w, h)
        want = cpu_render(lib, sb, cam, w, h)
        bitwise = float((util.bits(got) == util.bits(want)).all(axis=-1).mean())
        mse = float(((got.astype(np.float64) - want) ** 2).mean())
        psnr = 10.0 * np.log10(1.0 / mse) if mse > 0 else float("inf")
        print("%s %dx%d frame %d: %.4f of pixels bitwise equal, %.4f within 1e-4, %.1f dB" % (
            name, w, h, frame, bitwise, frac_within(got, want), psnr))
        assert want.max() > 0.1
        assert frac_within(got, want) >= 0.995
        assert psnr >= 36.0
    sc.release()


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h", CASES)
@pytest.mark.parametrize("group", [(8, 4), (16, 16)])
def test_tile_kernel_sees_its_work_group(ctx, oracle_dir, name, w, h, group):
    sb = util.scene(name)
    sc = ctx.upload(sb)
    pid = ctx.plugin_load(TILE)
    cam = util.default_camera()
    wb = (32, 16)
    got = ctx.render_plugin_cl(sc, cam, pid, w, h, kernel_mode=1, work_block=wb, group=group)
    want = cpu_render(cpu_oracle(TILE, oracle_dir), sb, cam, w, h, mode=1, work_block=wb, group=group)
    util.assert_bit_equal(got, want, "%s %dx%d group %s" % (name, w, h, group))
    with pytest.raises(capi.LtError):  # the file has no linearKernel
        ctx.render_plugin_cl(sc, cam, pid, w, h, kernel_mode=0, work_block=wb, group=group)
    sc.release()


@pytest.mark.gpu
def test_sizes_and_argument_errors(ctx, tmp_path):
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    cam = util.default_camera()
    p = tmp_path / "sizes.cl"
    p.write_text(SIZES + "__kernel void linearKernel(%s) {\n  if (get_global_id(0) + get_global_id(1) == 0) {\n"
                 "    output[0] = sizeof(float3); output[1] = sizeof(float4); output[2] = sizeof(uint3);\n  }\n}\n" % SIG)
    pid = ctx.plugin_load(str(p))
    got = ctx.render_plugin_cl(sc, cam, pid, 8, 4)
    assert got[0, 0].tolist() == [16.0, 16.0, 16.0]
    with pytest.raises(capi.LtError) as e:  # a group that does not divide the work block
        ctx.render_plugin_cl(sc, cam, pid, 64, 48, work_block=(24, 16), group=(16, 16))
    assert "-1" in str(e.value) and "divide" in str(e.value)
    with pytest.raises(capi.LtError) as e:  # an OpenCL C plug-in through the CUDA entry point
        ctx.render_plugin(sc, cam, pid, 8, 4)
    assert "-1" in str(e.value)
    cu = ctx.plugin_load(os.path.join(PLUGINS, "echo_buffers.cu"))
    with pytest.raises(capi.LtError) as e:  # and the other way round
        ctx.render_plugin_cl(sc, cam, cu, 8, 4)
    assert "-1" in str(e.value)
    with pytest.raises(capi.LtError) as e:
        ctx.plugin_load(os.path.join(PLUGINS, "does_not_exist.cl"))
    sc.release()


@pytest.mark.gpu
def test_renderer_opencl_runs_a_user_cl_file(ctx, tmp_path):
    """RendererOpenCL::render: MAX_FIT and a custom work block give what lt_render_plugin_cl gives; an edited copy
    shows the edit; a copy with a compile error leaves the buffer untouched."""
    os.chdir(util.ROOT)
    cam = host.Camera(0, 2.5, -50, 0)
    model = host.Model("resources/models/cornell_box_lens.obj")
    accel = host.AccelerationStructure(model)
    sb = accel.buffers()
    sc = ctx.upload(sb)
    pid = ctx.plugin_load(BARY)
    camera = util.default_camera()
    w, h = 101, 75
    r = host.Renderer(host.PLATFORM_OPENCL)
    util.assert_bit_equal(r.render(BARY, w, h, accel, model, cam), ctx.render_plugin_cl(sc, camera, pid, w, h))
    for mode in (0, 1):
        got = r.render(BARY, w, h, accel, model, cam, kernel_mode=mode, work_block=(25, 15), block=(5, 5))
        util.assert_bit_equal(got, ctx.render_plugin_cl(sc, camera, pid, w, h, kernel_mode=mode, work_block=(25, 15),
                                                        group=(5, 5)))
    text = open(BARY).read()
    store = "  output[id + 0] = colour.x;"
    assert store in text
    edited = tmp_path / "custom_opencl.cl"
    edited.write_text(text.replace(store, "  output[id + 0] = colour.x * 0.5f + 0.25f;"))
    assert capi.kernel_from_path(str(edited)) < 0
    got = r.render(str(edited), w, h, accel, model, cam)
    want = ctx.render_plugin_cl(sc, camera, pid, w, h)
    want[..., 0] = want[..., 0] * np.float32(0.5) + np.float32(0.25)
    util.assert_bit_equal(got, want, "edited colour store")
    broken = tmp_path / "broken.cl"
    broken.write_text(text.replace(store, "  output[id + 0] = colour.x"))
    out = np.full((h, w, 3), -1, np.float32)
    r.render(str(broken), w, h, accel, model, cam, out=out)
    assert (out == -1).all()
    sc.release()
    r.close()
    accel.close()
    model.close()
    cam.close()


@pytest.mark.gpu
def test_scene_file_names_a_user_cl_kernel(ctx, oracle_dir, tmp_path):
    os.chdir(util.ROOT)
    w, h = 96, 64
    scene = {"renderer": {"render_platform": "RENDER_PLATFORM_OPENCL", "kernel_file_path": BARY,
                          "kernel_mode": "KERNEL_MODE_LINEAR", "thread_organization_mode": "THREAD_ORGANIZATION_MODE_MAX_FIT",
                          "image_dimensions": [w, h, 3]},
             "camera": {"position": [0, 2.5, -50], "pitch": 0, "yaw": 0, "roll": 0},
             "world": {"cornell_box": {"file_path": "resources/models/cornell_box.obj"}},
             "output": {"file_path": str(tmp_path / "out.jpg")}}
    path = tmp_path / "user_cl.scene"
    path.write_text(json.dumps(scene))
    out = np.zeros((h, w, 3), np.float32)
    dims = (C.c_uint64 * 3)()
    rc = host.load().lth_run_scene_file(str(path).encode(), out.ctypes.data, out.nbytes, C.byref(dims))
    assert rc == 0 and tuple(dims) == (w, h, 3)
    want = cpu_render(cpu_oracle(BARY, oracle_dir), util.scene("cornell_box"), util.default_camera(), w, h)
    util.assert_bit_equal(out, want, "scene file")


# the reference's own .cl texts (vector-literal rewritten by oracle/build_ref_cl.sh, which leaves valid OpenCL C)
REF_TEXTS = [("basic", L.KERNEL_BASIC_CL, 0.998), ("custom_opencl", L.KERNEL_CUSTOM_BARY, 0.998),
             ("basic_lighting", L.KERNEL_LIGHTING25, 0.995), ("accumulator", L.KERNEL_ACCUMULATOR, 0.995),
             ("global_illumination_resources", L.KERNEL_GI25, 0.995),
             ("global_illumination_example", L.KERNEL_GI, 0.995)]


@pytest.mark.gpu
@pytest.mark.parametrize("stem,kernel,bound", REF_TEXTS, ids=[t[0] for t in REF_TEXTS])
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens"])
def test_reference_cl_texts_through_the_new_path(ctx, tmp_path, stem, kernel, bound, name):
    src = os.path.join(util.ROOT, "oracle", "_ref", "cl", stem + ".inc")
    if not os.path.exists(src):
        pytest.skip("oracle/_ref not built")
    path = tmp_path / (stem + ".cl")
    path.write_text(open(src).read())
    sb = util.scene(name)
    sc = ctx.upload(sb)
    pid = ctx.plugin_load(str(path))
    for frame in (0, 3):
        cam = util.default_camera(0.0, frame)
        got = ctx.render_plugin_cl(sc, cam, pid, 160, 120)
        want = ctx.render(sc, cam, capi.make_params(kernel, 160, 120))
        assert frac_within(got, want) >= bound, (stem, frame)
    sc.release()

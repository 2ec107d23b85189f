"""A/B against the REFERENCE ITSELF on the GPU box: oracle/_ref/libltref.so is the reference's own
Model / AccelerationStructureExplicit / RendererCUDA compiled from its sources (oracle/build_ref.sh);
RendererCUDA NVRTC-compiles its basic.cu exactly as shipped.  Identical in-memory buffers go to the
reference, to the new CUDA path and to the CPU oracle (the reference builder is nondeterministic, so
buffers are never compared across builders).

Without the reference's sources the live tests skip; the stored outputs of the reference's CUDA backend
(tests/golden/ref_cuda_*.npz, see tests/golden/README.md) keep the new CUDA path compared with it."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu

REF_DIR = os.path.join(util.ROOT, "oracle", "_ref")
REF_LIB = os.path.join(REF_DIR, "libltref.so")
KDIR = os.path.join(REF_DIR, "resources", "kernels", "cuda")


def _load_ref():
    if not os.path.exists(REF_LIB):
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    lib = C.CDLL(REF_LIB)
    vp, u64 = C.c_void_p, C.c_uint64
    for n in ("ltref_model_create", "ltref_as_create", "ltref_model_material_buffer", "ltref_as_node_buffer",
              "ltref_as_primitive_buffer", "ltref_as_light_buffer", "ltref_camera_create", "ltref_camera_buffer",
              "ltref_renderer_cuda_create"):
        getattr(lib, n).restype = vp
    for n in ("ltref_model_primitive_count", "ltref_model_material_bytes", "ltref_as_node_bytes",
              "ltref_as_primitive_bytes", "ltref_as_light_bytes"):
        getattr(lib, n).restype = u64
        getattr(lib, n).argtypes = [vp]
    lib.ltref_model_create.argtypes = [C.c_char_p]
    for n in ("ltref_as_create", "ltref_model_material_buffer", "ltref_as_node_buffer", "ltref_as_primitive_buffer",
              "ltref_as_light_buffer", "ltref_camera_buffer"):
        getattr(lib, n).argtypes = [vp]
    lib.ltref_camera_create.argtypes = [C.c_float] * 4
    lib.ltref_render_cuda.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, u64, u64, u64, u64, u64, vp, u64, vp, vp, vp]
    lib.ltref_render_cuda.restype = None
    return lib


class RefWorld:
    def __init__(self, lib, model_name):
        self.lib = lib
        path = os.path.join(REF_DIR, "resources", "models", model_name + ".obj")
        self.model = lib.ltref_model_create(path.encode())
        self.accel = lib.ltref_as_create(self.model)
        view = lambda p, n, dt: np.frombuffer((C.c_char * n).from_address(p), dtype=dt).copy()
        self.sb = L.SceneBuffers(
            view(lib.ltref_as_node_buffer(self.accel), lib.ltref_as_node_bytes(self.accel), L.NODE),
            view(lib.ltref_as_primitive_buffer(self.accel), lib.ltref_as_primitive_bytes(self.accel), L.PRIM),
            view(lib.ltref_model_material_buffer(self.model), lib.ltref_model_material_bytes(self.model), L.MATERIAL),
            view(lib.ltref_as_light_buffer(self.accel), lib.ltref_as_light_bytes(self.accel), L.LIGHTS))
        # the reference leaves the axis byte of leaves uninitialised; it is never read for leaves
        self.renderer = lib.ltref_renderer_cuda_create()

    def render(self, kernel_file, w, h, yaw=0.0, mode=0, block=None):
        cam = self.lib.ltref_camera_create(0, 2.5, -50, yaw)
        out = np.zeros((h, w, 3), np.float32)
        bx, by = block if block else (0, 0)
        self.lib.ltref_render_cuda(self.renderer, os.path.join(KDIR, kernel_file).encode(), mode, 1 if block else 0,
                                   bx, by, w, h, 3, out.ctypes.data, out.nbytes, self.accel, self.model, cam)
        return out


@pytest.fixture(scope="module")
def ref():
    return _load_ref()


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens"])
@pytest.mark.parametrize("yaw", [0.0, 0.03, -0.06, 0.25, 3.0])  # |yaw| < 0.1 keeps the model in view
def test_colour_and_hit_records_against_the_reference_cuda_backend(ref, ctx, name, yaw):
    world = RefWorld(ref, name)
    w, h = 256, 192
    cam = util.default_camera(yaw)
    sc = ctx.upload(world.sb)
    # colours: reference CUDA backend == new CUDA path == oracle, bit for bit
    ref_img = world.render("basic.cu", w, h, yaw)
    mine = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h))
    util.assert_bit_equal(mine, ref_img, "%s yaw %g: new CUDA path vs reference CUDA backend" % (name, yaw))
    util.assert_bit_equal(O.render(L.KERNEL_BASIC_CU, world.sb, cam, w, h, threads=0), ref_img,
                          "%s yaw %g: oracle vs reference CUDA backend" % (name, yaw))
    # tile mode and custom block through the reference give the same picture (its own invariants)
    util.assert_bit_equal(world.render("basic.cu", w, h, yaw, mode=1, block=(8, 8)), ref_img, "reference tile 8x8")
    if name != "cornell_box_lens":
        # hit records through the reference's own plugin mechanism (id_dump_*.cu = its traversal text
        # with the colour store replaced): primitive ids bit-exact, t/u/v bit-exact
        a = world.render("id_dump_a.cu", w, h, yaw)  # (id+1 as bits, t, u) on hit, zeros on miss
        b = world.render("id_dump_b.cu", w, h, yaw)  # (hitType+1 as bits, v, t)
        ref_hit = (b[..., 0].view(np.int32) == 2)
        ref_ids = a[..., 0].view(np.int32) - 1
        ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, w, h)
        np.testing.assert_array_equal(hit == 1, ref_hit)
        np.testing.assert_array_equal(ids[ref_hit], ref_ids[ref_hit])
        util.assert_bit_equal(tuv[..., 0][ref_hit], a[..., 1][ref_hit], "t")
        util.assert_bit_equal(tuv[..., 1][ref_hit], a[..., 2][ref_hit], "u")
        util.assert_bit_equal(tuv[..., 2][ref_hit], b[..., 1][ref_hit], "v")
    sc.release()


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(util.GOLDEN, "ref_cuda_*.npz"))),
                         ids=lambda p: os.path.basename(p)[9:-4])
def test_colour_and_hit_records_against_the_reference_golden(ctx, path):
    """The reference's CUDA backend output stored with the buffers its builder made: the new CUDA path renders
    the same picture and finds the same primary hits, bit for bit."""
    z = np.load(path)
    sb = L.SceneBuffers(z["nodes"], z["prims"], z["materials"], z["lights"])
    cam = z["camera"].view(L.CAMERA)
    w, h = int(z["width"]), int(z["height"])
    sc = ctx.upload(sb)
    mine = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h))
    util.assert_bit_equal(mine, z["color"], os.path.basename(path) + ": new CUDA path vs reference CUDA backend")
    if "ids" in z:
        ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, w, h)
        m = z["hit"] == 1
        np.testing.assert_array_equal(hit, z["hit"])
        np.testing.assert_array_equal(ids[m], z["ids"][m])
        util.assert_bit_equal(tuv[m], z["tuv"][m], os.path.basename(path) + " t,u,v")
    sc.release()


def test_model_loader_matches_the_reference_loader(ref):
    """This repo's OBJ/MTL reader vs the reference's (tinyobjloader): same triangles, normals,
    materials, for the reference's original asset files and for this repo's canonical re-emits."""
    from lens_trace_b200 import host
    for name in ("green_wall", "cornell_box", "cornell_box_lens"):
        world = RefWorld(ref, name)
        for path in (os.path.join(REF_DIR, "resources", "models", name + ".obj"),
                     os.path.join(util.MODELS, name + ".obj")):
            sb = host.load_scene_buffers(path)
            key = lambda p: p.tobytes()
            assert sorted(map(key, sb.prims)) == sorted(map(key, world.sb.prims)), (name, path)
            assert sb.materials.tobytes() == world.sb.materials.tobytes()

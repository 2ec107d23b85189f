"""ctypes binding of the C++ host surface (liblenstrace.so, include/lens_trace/b200/host_capi.h):
Model, AccelerationStructureExplicit, Camera, RendererCUDA/RendererOpenCL -- the objects the reference's
examples and tests construct (tests/cuda_renderer_test.cc:12-49)."""
import ctypes as C
import os

import numpy as np

from . import layouts as L

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblenstrace.so")

PLATFORM_OPENCL = 0
PLATFORM_CUDA = 1

SYMBOLS = [
    "lth_model_create", "lth_model_destroy", "lth_model_ok", "lth_model_primitive_count", "lth_model_material_buffer",
    "lth_model_material_bytes", "lth_as_create", "lth_as_create_typed", "lth_as_destroy", "lth_as_node_buffer", "lth_as_node_bytes",
    "lth_as_primitive_buffer", "lth_as_primitive_bytes", "lth_as_light_buffer", "lth_as_light_bytes",
    "lth_camera_create", "lth_camera_destroy", "lth_camera_buffer", "lth_camera_set_frame_count",
    "lth_camera_increment_frame_count", "lth_camera_set_position", "lth_camera_set_rotation", "lth_renderer_create",
    "lth_renderer_destroy", "lth_renderer_cached_scenes", "lth_render", "lth_write_synthetic_scene", "lth_run_scene_file",
]


class RenderExtensionB200(C.Structure):
    _fields_ = [
        ("sType", C.c_int), ("pNext", C.c_void_p), ("frames", C.c_uint32), ("accumulate", C.c_uint32),
        ("maxRayDepth", C.c_uint32), ("collectStats", C.c_uint32), ("rays", C.c_uint64), ("nodeTests", C.c_uint64),
        ("triTests", C.c_uint64), ("kernelMilliseconds", C.c_float), ("deviceCount", C.c_uint32),
        ("splitMode", C.c_uint32),
    ]


STRUCTURE_TYPE_RENDER_EXTENSION_B200 = 1000

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("liblenstrace.so is not built: run `python -m lens_trace_b200.build`")
    lib = C.CDLL(LIB_PATH)
    vp, u64 = C.c_void_p, C.c_uint64
    for name in ("lth_model_create", "lth_as_create", "lth_model_material_buffer", "lth_as_node_buffer",
                 "lth_as_primitive_buffer", "lth_as_light_buffer", "lth_camera_buffer", "lth_camera_create",
                 "lth_renderer_create"):
        getattr(lib, name).restype = vp
    for name in ("lth_model_primitive_count", "lth_model_material_bytes", "lth_as_node_bytes",
                 "lth_as_primitive_bytes", "lth_as_light_bytes", "lth_write_synthetic_scene"):
        getattr(lib, name).restype = u64
    lib.lth_model_create.argtypes = [C.c_char_p]
    for name in ("lth_model_destroy", "lth_model_ok", "lth_model_primitive_count", "lth_model_material_buffer",
                 "lth_model_material_bytes", "lth_as_create", "lth_as_create_typed", "lth_as_destroy", "lth_as_node_buffer",
                 "lth_as_node_bytes", "lth_as_primitive_buffer", "lth_as_primitive_bytes", "lth_as_light_buffer",
                 "lth_as_light_bytes", "lth_camera_destroy", "lth_camera_buffer", "lth_camera_increment_frame_count"):
        getattr(lib, name).argtypes = [vp]
    lib.lth_as_create_typed.restype = vp
    lib.lth_as_create_typed.argtypes = [vp, C.c_int]
    lib.lth_camera_create.argtypes = [C.c_float] * 4
    lib.lth_camera_set_frame_count.argtypes = [vp, C.c_uint32]
    lib.lth_camera_set_position.argtypes = [vp, C.c_float, C.c_float, C.c_float]
    lib.lth_camera_set_rotation.argtypes = [vp, C.c_float, C.c_float, C.c_float]
    lib.lth_renderer_create.argtypes = [C.c_int]
    lib.lth_renderer_destroy.argtypes = [vp, C.c_int]
    lib.lth_renderer_cached_scenes.argtypes = [vp, C.c_int]
    lib.lth_renderer_cached_scenes.restype = C.c_uint64
    lib.lth_render.argtypes = [vp, C.c_int, C.c_char_p, C.c_int, C.c_int, u64, u64, u64, u64, u64, vp, u64, vp, vp, vp,
                               vp]
    lib.lth_render.restype = None
    lib.lth_write_synthetic_scene.argtypes = [C.c_char_p, C.c_uint32, u64]
    lib.lth_run_scene_file.argtypes = [C.c_char_p, vp, u64, C.POINTER(u64 * 3)]
    _lib = lib
    return lib


def _view(ptr, nbytes, dtype):
    buf = (C.c_char * nbytes).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype)


class Model:
    def __init__(self, path):
        self.lib = load()
        self.h = self.lib.lth_model_create(path.encode())

    @property
    def primitive_count(self):
        return self.lib.lth_model_primitive_count(self.h)

    def materials(self):
        n = self.lib.lth_model_material_bytes(self.h)
        return _view(self.lib.lth_model_material_buffer(self.h), n, L.MATERIAL).copy() if n else np.zeros(0, L.MATERIAL)

    def close(self):
        if self.h:
            self.lib.lth_model_destroy(self.h)
            self.h = None


class AccelerationStructure:
    HOST_MEDIAN_SPLIT = 0
    GPU_LBVH = 100
    HOST_SAH = 101
    GPU_PLOC = 102

    def __init__(self, model, kind=0):
        self.lib = load()
        self.model = model
        self.h = self.lib.lth_as_create_typed(model.h, kind)

    def buffers(self):
        """Copies of the flat buffers as layouts.SceneBuffers."""
        lib = self.lib
        nodes = _view(lib.lth_as_node_buffer(self.h), lib.lth_as_node_bytes(self.h), L.NODE).copy()
        prims = _view(lib.lth_as_primitive_buffer(self.h), lib.lth_as_primitive_bytes(self.h), L.PRIM).copy()
        lights = _view(lib.lth_as_light_buffer(self.h), lib.lth_as_light_bytes(self.h), L.LIGHTS).copy()
        return L.SceneBuffers(nodes, prims, self.model.materials(), lights)

    def close(self):
        if self.h:
            self.lib.lth_as_destroy(self.h)
            self.h = None


class Camera:
    def __init__(self, x, y, z, yaw=0.0):
        self.lib = load()
        self.h = self.lib.lth_camera_create(x, y, z, yaw)

    def buffer(self):
        return _view(self.lib.lth_camera_buffer(self.h), 28, L.CAMERA).copy()

    def set_frame_count(self, n):
        self.lib.lth_camera_set_frame_count(self.h, n)

    def increment_frame_count(self):
        self.lib.lth_camera_increment_frame_count(self.h)

    def close(self):
        if self.h:
            self.lib.lth_camera_destroy(self.h)
            self.h = None


class Renderer:
    """RendererCUDA (platform=1) or RendererOpenCL (platform=0) of include/lens_trace/."""

    def __init__(self, platform=PLATFORM_CUDA):
        self.lib = load()
        self.platform = platform
        self.h = self.lib.lth_renderer_create(platform)

    def render(self, kernel_file_path, width, height, accel, model, camera, depth=3, kernel_mode=0, block=None,
               ext=None, out=None):
        if out is None:
            out = np.zeros((height, width, depth), dtype=np.float32)
        bx, by = block if block else (0, 0)
        self.lib.lth_render(self.h, self.platform, kernel_file_path.encode(), kernel_mode, 1 if block else 0, bx, by,
                            width, height, depth, out.ctypes.data, out.nbytes, accel.h, model.h, camera.h,
                            C.addressof(ext) if ext is not None else None)
        return out

    def cached_scenes(self):
        return int(self.lib.lth_renderer_cached_scenes(self.h, self.platform))

    def close(self):
        if self.h:
            self.lib.lth_renderer_destroy(self.h, self.platform)
            self.h = None


def make_extension(frames=1, accumulate=False, max_ray_depth=0, collect_stats=False, devices=0, split=0):
    e = RenderExtensionB200()
    e.sType = STRUCTURE_TYPE_RENDER_EXTENSION_B200
    e.pNext = None
    e.frames, e.accumulate, e.maxRayDepth, e.collectStats = frames, int(accumulate), max_ray_depth, int(collect_stats)
    e.deviceCount, e.splitMode = devices, split
    return e


def write_synthetic_scene(path, grid_n, seed=0x5EED):
    n = load().lth_write_synthetic_scene(path.encode(), grid_n, seed)
    if n == 0:
        raise RuntimeError("cannot write synthetic scene to %s" % path)
    return n


def load_scene_buffers(obj_path, kind=0):
    """OBJ -> Model -> AccelerationStructureExplicit (kind: 0 median split, 100 GPU LBVH, 101 host SAH,
    102 GPU PLOC) -> flat
    buffers (layouts.SceneBuffers)."""
    m = Model(obj_path)
    if m.primitive_count == 0:
        m.close()
        raise RuntimeError("model %s has no primitives" % obj_path)
    a = AccelerationStructure(m, kind)
    sb = a.buffers()
    a.close()
    m.close()
    return sb

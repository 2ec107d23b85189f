"""ctypes binding of the C-ABI in include/lens_trace_b200.h (liblt_b200.so).

This is the same set of calls a maintainer of the reference would bind from
src/cuda/renderer_cuda.cpp (INTEGRATION.md).  Nothing here computes: if the library is missing or no
CUDA device is usable, calls raise LtError -- there is no fallback path.
"""
import ctypes as C
import os

import numpy as np

from . import layouts as L

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblt_b200.so")

SYMBOLS = [
    "lt_api_version", "lt_ctx_create", "lt_ctx_destroy", "lt_last_error", "lt_ctx_set_stream", "lt_scene_upload",
    "lt_scene_release", "lt_render", "lt_render_device", "lt_accum_reset", "lt_accum_read", "lt_primary_hits",
    "lt_last_stats", "lt_kernel_from_path", "lt_kernel_name", "lt_debug_random", "lt_debug_hemisphere", "lt_debug_build_threaded", "lt_debug_build_threaded_pruned", "lt_debug_scene_full_threaded", "lt_plugin_load", "lt_render_plugin", "lt_primary_hits_flags", "lt_scene_build_lbvh", "lt_scene_build_ploc", "lt_scene_download", "lt_scene_info",
    "lt_debug_gather_peak", "lt_ctx_create_multi", "lt_ctx_device_count", "lt_host_register", "lt_host_unregister", "lt_debug_tile_rows",
]


class LtError(RuntimeError):
    pass


class RenderParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("kernel", C.c_int32), ("kernel_mode", C.c_int32), ("width", C.c_int32),
        ("height", C.c_int32), ("depth", C.c_int32), ("max_ray_depth", C.c_int32), ("frames", C.c_int32),
        ("frame_stride", C.c_uint32), ("accum_mode", C.c_int32), ("accum_weight", C.c_float), ("flags", C.c_int32),
        ("block_x", C.c_int32), ("block_y", C.c_int32), ("split_mode", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("rays", C.c_uint64), ("node_tests", C.c_uint64), ("tri_tests", C.c_uint64), ("kernel_ms", C.c_float),
        ("upload_ms", C.c_float), ("kernel_launches", C.c_int32), ("sm_count", C.c_int32), ("trace_ms", C.c_float),
        ("trace_launches", C.c_int32), ("shade_ms", C.c_float), ("primary_shade_ms", C.c_float),
        ("accumulate_ms", C.c_float), ("shade_launches", C.c_int32),
    ]


_lib = None


def load():
    """Loads liblt_b200.so (no CUDA call is made by loading)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LtError("liblt_b200.so is not built: run `python -m lens_trace_b200.build` (there is no fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.lt_api_version.restype = C.c_int
    lib.lt_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.lt_ctx_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
    lib.lt_ctx_device_count.argtypes = [C.c_void_p]
    lib.lt_host_register.argtypes = [C.c_void_p, C.c_uint64]
    lib.lt_host_unregister.argtypes = [C.c_void_p]
    lib.lt_debug_tile_rows.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    lib.lt_ctx_destroy.argtypes = [C.c_void_p]
    lib.lt_ctx_destroy.restype = None
    lib.lt_last_error.argtypes = [C.c_void_p]
    lib.lt_last_error.restype = C.c_char_p
    lib.lt_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.lt_scene_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                    C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.lt_scene_build_lbvh.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.lt_scene_build_ploc.argtypes = lib.lt_scene_build_lbvh.argtypes
    lib.lt_scene_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.lt_scene_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]
    lib.lt_scene_release.argtypes = [C.c_void_p, C.c_void_p]
    lib.lt_scene_release.restype = None
    lib.lt_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams), C.c_void_p]
    lib.lt_render_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams), C.c_void_p, C.c_int]
    lib.lt_accum_reset.argtypes = [C.c_void_p]
    lib.lt_accum_read.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    lib.lt_primary_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    lib.lt_primary_hits_flags.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lt_last_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    lib.lt_debug_random.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.lt_debug_hemisphere.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.lt_debug_build_threaded.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    lib.lt_debug_build_threaded_pruned.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_int32)]
    lib.lt_debug_scene_full_threaded.argtypes = [C.c_void_p, C.c_int]
    lib.lt_plugin_load.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_int)]
    lib.lt_render_plugin.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_void_p]
    lib.lt_debug_gather_peak.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.lt_kernel_from_path.argtypes = [C.c_char_p]
    lib.lt_kernel_name.argtypes = [C.c_int]
    lib.lt_kernel_name.restype = C.c_char_p
    _lib = lib
    return lib


def kernel_from_path(path):
    return load().lt_kernel_from_path(path.encode())


def make_params(kernel, width, height, depth=3, kernel_mode=0, max_ray_depth=0, frames=1, frame_stride=1,
                accum_mode=L.ACCUM_NONE, accum_weight=0.0, flags=0, split_mode=0):
    p = RenderParams()
    p.struct_size = C.sizeof(RenderParams)
    p.kernel, p.kernel_mode = kernel, kernel_mode
    p.width, p.height, p.depth = width, height, depth
    p.max_ray_depth, p.frames, p.frame_stride = max_ray_depth, frames, frame_stride
    p.accum_mode, p.accum_weight, p.flags = accum_mode, accum_weight, flags
    p.split_mode = split_mode
    return p


class Context:
    """lt_ctx: one per GPU, or -- device = a list of ordinals -- one multi-GPU context (lt_ctx_create_multi)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            arr = (C.c_int * len(device))(*device)
            rc = self.lib.lt_ctx_create_multi(arr, len(device), C.byref(h))
        else:
            rc = self.lib.lt_ctx_create(device, C.byref(h))
        if rc != 0:
            raise LtError("lt_ctx_create failed (%d): %s" % (rc, self.lib.lt_last_error(None).decode()))
        self.h = h

    def device_count(self):
        return self.lib.lt_ctx_device_count(self.h)

    def close(self):
        if self.h:
            self.lib.lt_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc != 0:
            raise LtError("%s failed (%d): %s" % (what, rc, self.lib.lt_last_error(self.h).decode()))

    def set_stream(self, cuda_stream_ptr):
        self._check(self.lib.lt_ctx_set_stream(self.h, C.c_void_p(cuda_stream_ptr)), "lt_ctx_set_stream")

    def upload(self, scene):
        """scene: layouts.SceneBuffers -> Scene handle"""
        out = C.c_void_p()
        rc = self.lib.lt_scene_upload(self.h, scene.nodes.ctypes.data, scene.nodes.nbytes, scene.prims.ctypes.data,
                                      scene.prims.nbytes, scene.materials.ctypes.data, scene.materials.nbytes,
                                      scene.lights.ctypes.data, scene.lights.nbytes, C.byref(out))
        self._check(rc, "lt_scene_upload")
        return Scene(self, out)

    def build_lbvh(self, prims, materials):
        """Device-side LBVH over `prims` (layouts.PRIM array in any order) -> Scene handle"""
        return self._build("lt_scene_build_lbvh", prims, materials)

    def build_ploc(self, prims, materials):
        """Device-side PLOC tree over `prims` (layouts.PRIM array in any order) -> Scene handle"""
        return self._build("lt_scene_build_ploc", prims, materials)

    def _build(self, entry, prims, materials):
        prims = np.ascontiguousarray(prims, dtype=L.PRIM)
        materials = np.ascontiguousarray(materials, dtype=L.MATERIAL)
        out = C.c_void_p()
        rc = getattr(self.lib, entry)(self.h, prims.ctypes.data, prims.nbytes, materials.ctypes.data, materials.nbytes,
                                      C.byref(out))
        self._check(rc, entry)
        sc = Scene(self, out)
        sc.materials = materials.copy()
        return sc

    def download(self, scene):
        """The scene's buffers in the reference layouts (layouts.SceneBuffers); materials as uploaded."""
        nn, np_, sd = C.c_uint64(), C.c_uint64(), C.c_int32()
        self.lib.lt_scene_info(scene.h, C.byref(nn), C.byref(np_), C.byref(sd))
        nodes = np.zeros(nn.value, dtype=L.NODE)
        prims = np.zeros(np_.value, dtype=L.PRIM)
        lights = np.zeros(1, dtype=L.LIGHTS)
        self._check(self.lib.lt_scene_download(self.h, scene.h, nodes.ctypes.data, nodes.nbytes, prims.ctypes.data,
                                               prims.nbytes, lights.ctypes.data), "lt_scene_download")
        return L.SceneBuffers(nodes, prims, getattr(scene, "materials", np.zeros(0, L.MATERIAL)), lights), sd.value

    def render(self, scene, camera, params, want_output=True):
        """Host-buffer path (lt_render): returns float32 [H, W, depth] or None."""
        out = None
        ptr = None
        if want_output:
            out = np.empty((params.height, params.width, params.depth), dtype=np.float32)
            ptr = out.ctypes.data
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render(self.h, scene.h, cam.ctypes.data, C.byref(params), ptr), "lt_render")
        return out

    def render_into(self, scene, camera, params, host_ptr):
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render(self.h, scene.h, cam.ctypes.data, C.byref(params), C.c_void_p(host_ptr)),
                    "lt_render")

    def render_device(self, scene, camera, params, device_ptr, sync=False):
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_device(self.h, scene.h, cam.ctypes.data, C.byref(params),
                                              C.c_void_p(device_ptr), 1 if sync else 0), "lt_render_device")

    def accum_reset(self):
        self._check(self.lib.lt_accum_reset(self.h), "lt_accum_reset")

    def primary_hits(self, scene, camera, kernel, width, height, flags=0):
        ids = np.empty((height, width), dtype=np.int32)
        hit = np.empty((height, width), dtype=np.int32)
        tuv = np.empty((height, width, 3), dtype=np.float32)
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_primary_hits_flags(self.h, scene.h, cam.ctypes.data, kernel, flags, width, height,
                                                   ids.ctypes.data, hit.ctypes.data, tuv.ctypes.data),
                    "lt_primary_hits_flags")
        return ids, hit, tuv

    def plugin_load(self, path):
        pid = C.c_int(-1)
        self._check(self.lib.lt_plugin_load(self.h, path.encode(), C.byref(pid)), "lt_plugin_load")
        return pid.value

    def render_plugin(self, scene, camera, plugin_id, width, height, depth=3, kernel_mode=0, block=(0, 0)):
        out = np.zeros((height, width, depth), dtype=np.float32)
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_plugin(self.h, scene.h, cam.ctypes.data, plugin_id, kernel_mode, width, height,
                                              depth, block[0], block[1], out.ctypes.data), "lt_render_plugin")
        return out

    def debug_random(self, fx, fy, seed):
        fx, fy, seed = (np.ascontiguousarray(a, dtype=np.float32) for a in (fx, fy, seed))
        out = np.empty_like(fx)
        self._check(self.lib.lt_debug_random(self.h, fx.ctypes.data, fy.ctypes.data, seed.ctypes.data, fx.size,
                                             out.ctypes.data), "lt_debug_random")
        return out

    def debug_hemisphere(self, u1, u2, up):
        u1, u2, up = (np.ascontiguousarray(a, dtype=np.float32) for a in (u1, u2, up))
        out = np.empty((u1.size, 4), dtype=np.float32)
        self._check(self.lib.lt_debug_hemisphere(self.h, u1.ctypes.data, u2.ctypes.data, up.ctypes.data, u1.size,
                                                 out.ctypes.data), "lt_debug_hemisphere")
        return out

    def gather_peak(self, table_bytes, dependent=False, ilp=4, blocks_per_sm=8, iters=2000):
        """(GB/s, ns per gather and lane) of per-lane 32-byte gathers on a table of table_bytes"""
        gbs, ns = C.c_double(0.0), C.c_double(0.0)
        self._check(self.lib.lt_debug_gather_peak(self.h, int(table_bytes), 1 if dependent else 0, ilp, blocks_per_sm,
                                                  iters, C.byref(gbs), C.byref(ns)), "lt_debug_gather_peak")
        return gbs.value, ns.value

    def debug_full_threaded(self, scene, full):
        """Test hook: every ray of later launches on `scene` walks the full threaded copies (full=True), or rays
        with finite, nonzero reciprocals walk the pruned ones again (full=False, the default after upload)."""
        self._check(self.lib.lt_debug_scene_full_threaded(scene.h, 1 if full else 0), "lt_debug_scene_full_threaded")

    def stats(self):
        s = Stats()
        self.lib.lt_last_stats(self.h, C.byref(s))
        return s


class Scene:
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    def release(self):
        if self.h and self.ctx.h:
            self.ctx.lib.lt_scene_release(self.ctx.h, self.h)
        self.h = None


def tile_rows(height, devices, device):
    """Host-only: image rows device `device` of `devices` renders in a tile split, in local-row order."""
    lib = load()
    n = lib.lt_debug_tile_rows(height, devices, device, None, 0)
    if n < 0:
        raise LtError("lt_debug_tile_rows: bad arguments")
    out = np.zeros(n, np.int32)
    lib.lt_debug_tile_rows(height, devices, device, out.ctypes.data, n)
    return out


THREAD_NODE = np.dtype([("lo", "<f4", 3), ("hix", "<f4"), ("hiy", "<f4"), ("hiz", "<f4"), ("link", "<i4"), ("skip", "<i4")])


def build_threaded(nodes):
    """Host-only: the 8 x N threaded records lt_scene_upload builds for small trees (lt_debug_build_threaded)."""
    lib = load()
    nodes = np.ascontiguousarray(nodes)
    out = np.zeros((8, len(nodes)), THREAD_NODE)
    rc = lib.lt_debug_build_threaded(nodes.ctypes.data, nodes.nbytes, out.ctypes.data)
    if rc != 0:
        raise LtError("lt_debug_build_threaded failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    return out


def build_threaded_pruned(nodes):
    """Host-only: the 8 x stride pruned threaded records lt_scene_upload builds beside the full ones
    (lt_debug_build_threaded_pruned); skip links index the returned array flattened."""
    lib = load()
    nodes = np.ascontiguousarray(nodes)
    stride = C.c_int32(0)
    out = np.zeros((8, len(nodes)), THREAD_NODE)
    rc = lib.lt_debug_build_threaded_pruned(nodes.ctypes.data, nodes.nbytes, out.ctypes.data, C.byref(stride))
    if rc != 0:
        raise LtError("lt_debug_build_threaded_pruned failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    return np.ascontiguousarray(out.reshape(-1)[:8 * stride.value].reshape(8, stride.value))

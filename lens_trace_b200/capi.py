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
    "lt_last_stats", "lt_kernel_from_path", "lt_kernel_name", "lt_debug_random", "lt_debug_hemisphere", "lt_debug_build_threaded", "lt_debug_build_threaded_pruned", "lt_debug_scene_full_threaded", "lt_plugin_load", "lt_render_plugin", "lt_render_plugin_cl", "lt_debug_compile_cl", "lt_debug_translate_cl", "lt_primary_hits_flags", "lt_scene_build_lbvh", "lt_scene_build_ploc", "lt_scene_download", "lt_scene_info",
    "lt_debug_gather_peak", "lt_ctx_create_multi", "lt_ctx_device_count", "lt_host_register", "lt_host_unregister", "lt_debug_tile_rows",
    "lt_debug_plan", "lt_debug_ctx_limits", "lt_render_plugin_frames", "lt_debug_build_traversal_tree",
    "lt_debug_scene_traversal_tree", "lt_debug_traversal_tree", "lt_render_views", "lt_render_views_device",
    "lt_debug_plan_views", "lt_scene_refit", "lt_scene_refit_device", "lt_debug_scene_bytes",
    "lt_render_masked_device", "lt_debug_plan_masked", "lt_debug_ctx_list_order", "lt_render_adaptive",
    "lt_render_adaptive_device", "lt_debug_adaptive_rounds", "lt_debug_ctx_adaptive_part",
    "lt_debug_ctx_create_shared",
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


class AdaptiveParams(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("target", C.c_float), ("floor", C.c_float), ("round_frames", C.c_int32),
                ("max_frames", C.c_int32)]


class AdaptiveResult(C.Structure):
    _fields_ = [("rounds", C.c_int32), ("pixel_frames", C.c_uint64), ("pixels_unconverged", C.c_uint64)]


def make_adaptive(target, max_frames, round_frames=0, floor=0.0):
    a = AdaptiveParams()
    a.struct_size = C.sizeof(AdaptiveParams)
    a.target, a.floor, a.round_frames, a.max_frames = target, floor, round_frames, max_frames
    return a


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
    lib.lt_debug_ctx_create_shared.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_void_p)]
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
    lib.lt_scene_refit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.lt_scene_refit_device.argtypes = lib.lt_scene_refit.argtypes
    lib.lt_scene_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]
    lib.lt_scene_release.argtypes = [C.c_void_p, C.c_void_p]
    lib.lt_scene_release.restype = None
    lib.lt_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams), C.c_void_p]
    lib.lt_render_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams), C.c_void_p, C.c_int]
    lib.lt_render_views.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(RenderParams), C.c_void_p]
    lib.lt_render_views_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(RenderParams),
                                           C.c_void_p, C.c_int]
    lib.lt_render_masked_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams), C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_int]
    lib.lt_debug_ctx_list_order.argtypes = [C.c_void_p, C.c_int]
    lib.lt_render_adaptive.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams),
                                       C.POINTER(AdaptiveParams), C.c_void_p, C.c_void_p, C.POINTER(AdaptiveResult)]
    lib.lt_render_adaptive_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderParams),
                                              C.POINTER(AdaptiveParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.POINTER(AdaptiveResult), C.c_int]
    lib.lt_debug_adaptive_rounds.argtypes = [C.POINTER(RenderParams), C.POINTER(AdaptiveParams), C.c_uint32, C.c_void_p,
                                             C.c_int]
    lib.lt_debug_ctx_adaptive_part.argtypes = [C.c_void_p, C.c_int, C.c_int]
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
    lib.lt_debug_build_traversal_tree.argtypes = [C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p, C.POINTER(C.c_int32),
                                                  C.c_void_p, C.POINTER(C.c_int32)]
    lib.lt_debug_scene_traversal_tree.argtypes = [C.c_void_p]
    lib.lt_debug_scene_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.lt_debug_traversal_tree.argtypes = [C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p, C.POINTER(C.c_double)]
    lib.lt_debug_ctx_limits.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.lt_debug_plan.argtypes = [C.POINTER(RenderParams), C.c_uint64, C.c_int32, C.c_uint64, C.c_int32,
                                  C.POINTER(C.c_int64)]
    lib.lt_debug_plan_views.argtypes = [C.POINTER(RenderParams), C.c_int, C.c_uint64, C.c_int32, C.c_uint64, C.c_int32,
                                        C.POINTER(C.c_int64)]
    lib.lt_debug_plan_masked.argtypes = [C.POINTER(RenderParams), C.c_int64, C.c_uint64, C.c_int32, C.c_uint64,
                                         C.c_int32, C.POINTER(C.c_int64)]
    lib.lt_plugin_load.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_int)]
    lib.lt_render_plugin.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_void_p]
    lib.lt_render_plugin_cl.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 9 + [C.c_void_p]
    lib.lt_render_plugin_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(RenderParams), C.c_int,
                                            C.c_int, C.c_void_p]
    lib.lt_debug_compile_cl.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64]
    lib.lt_debug_translate_cl.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64, C.POINTER(C.c_int32)]
    lib.lt_debug_translate_cl.restype = C.c_int64
    lib.lt_debug_gather_peak.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.lt_kernel_from_path.argtypes = [C.c_char_p]
    lib.lt_kernel_name.argtypes = [C.c_int]
    lib.lt_kernel_name.restype = C.c_char_p
    _lib = lib
    return lib


def kernel_from_path(path):
    return load().lt_kernel_from_path(path.encode())


def compile_cl(path, log_bytes=1 << 20):
    """Translate and compile an OpenCL C kernel file for sm_100a as lt_plugin_load would, without a device.
    Returns (ok, log): the log holds the reason or the NVRTC messages, which name the file and line."""
    log = C.create_string_buffer(log_bytes)
    rc = load().lt_debug_compile_cl(path.encode(), log, log_bytes)
    return rc == 0, log.value.decode(errors="replace")


def translate_cl(text):
    """The library's translation of OpenCL C text (see lt_debug_translate_cl): (translated text, contraction off)."""
    lib = load()
    off = C.c_int32(0)
    n = lib.lt_debug_translate_cl(text.encode(), None, 0, C.byref(off))
    buf = C.create_string_buffer(n)
    lib.lt_debug_translate_cl(text.encode(), buf, n, C.byref(off))
    return buf.value.decode(), bool(off.value)


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
        self.shared_device = None

    @classmethod
    def shared(cls, device, members):
        """Test hook (lt_debug_ctx_create_shared): a multi-device Context of `members` members that all render on
        `device`; shared_device is then that ordinal (None on every other Context)."""
        self = cls.__new__(cls)
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.lt_debug_ctx_create_shared(device, members, C.byref(h))
        if rc != 0:
            raise LtError("lt_debug_ctx_create_shared failed (%d): %s" % (rc, self.lib.lt_last_error(None).decode()))
        self.h = h
        self.shared_device = device
        return self

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

    def refit(self, scene, prims):
        """Replace the scene's primitives (layouts.PRIM array in the order of its primitive buffer) and refit its tree
        on the device (lt_scene_refit); the topology, materials and lights stay."""
        prims = np.ascontiguousarray(prims, dtype=L.PRIM)
        self._check(self.lib.lt_scene_refit(self.h, scene.h, prims.ctypes.data, prims.nbytes), "lt_scene_refit")

    def refit_device(self, scene, device_ptr, nbytes):
        """lt_scene_refit_device: the new primitives are nbytes of device memory at device_ptr (e.g. a torch CUDA
        tensor's data_ptr())"""
        self._check(self.lib.lt_scene_refit_device(self.h, scene.h, C.c_void_p(device_ptr), nbytes),
                    "lt_scene_refit_device")

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

    def render_views(self, scene, cameras, params, want_output=True):
        """Several views in one call (lt_render_views): cameras is a sequence of V camera records; returns float32
        [V, H, W, depth] (view v equals accum_reset + render of camera v) or None."""
        cams = np.ascontiguousarray(cameras, dtype=L.CAMERA).reshape(-1)
        out = None
        if want_output:
            out = np.empty((cams.size, params.height, params.width, params.depth), dtype=np.float32)
        self._check(self.lib.lt_render_views(self.h, scene.h, cams.ctypes.data if cams.size else None, cams.size,
                                             C.byref(params), out.ctypes.data if out is not None else None),
                    "lt_render_views")
        return out

    def render_views_device(self, scene, cameras, params, device_ptr, sync=False):
        """lt_render_views_device: V images at device_ptr (V * H * W * depth floats), slice v the accumulator of view v"""
        cams = np.ascontiguousarray(cameras, dtype=L.CAMERA).reshape(-1)
        self._check(self.lib.lt_render_views_device(self.h, scene.h, cams.ctypes.data if cams.size else None, cams.size,
                                                    C.byref(params), C.c_void_p(device_ptr), 1 if sync else 0),
                    "lt_render_views_device")

    def render_masked_device(self, scene, camera, params, out_ptr, mask_ptr=None, m2_ptr=None, sync=False):
        """lt_render_masked_device: lt_render_device for the pixels whose byte of the H x W uint8 mask at mask_ptr is
        nonzero (None: every pixel); pixels outside the mask are not written.  m2_ptr: H * W * 3 floats of Welford sums
        beside a running mean (None: not kept).  All pointers are device memory of the context's device, e.g. torch
        CUDA tensors' data_ptr()."""
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_masked_device(self.h, scene.h, cam.ctypes.data, C.byref(params),
                                                     C.c_void_p(mask_ptr) if mask_ptr else None, C.c_void_p(out_ptr),
                                                     C.c_void_p(m2_ptr) if m2_ptr else None, 1 if sync else 0),
                    "lt_render_masked_device")

    def render_adaptive(self, scene, camera, params, target, round_frames=0, max_frames=None, floor=0.0):
        """lt_render_adaptive: params.frames frames on every pixel, then rounds of round_frames (0: params.frames) on
        the pixels whose relative standard error is still above target, up to max_frames (None: params.frames + 3
        rounds).  Returns (mean float32 [H, W, depth], frame counts uint32 [H, W], AdaptiveResult)."""
        if max_frames is None:
            max_frames = params.frames + 3 * (round_frames or params.frames)
        a = make_adaptive(target, max_frames, round_frames, floor)
        out = np.empty((params.height, params.width, params.depth), dtype=np.float32)
        frames = np.empty((params.height, params.width), dtype=np.uint32)
        res = AdaptiveResult()
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_adaptive(self.h, scene.h, cam.ctypes.data, C.byref(params), C.byref(a),
                                                out.ctypes.data, frames.ctypes.data, C.byref(res)), "lt_render_adaptive")
        return out, frames, res

    def render_adaptive_device(self, scene, camera, params, out_ptr, m2_ptr, frames_ptr=None, target=0.05,
                               round_frames=0, max_frames=None, floor=0.0, sync=False):
        """lt_render_adaptive_device: the adaptive loop continued in device memory -- out_ptr (H * W * depth floats of
        running mean), m2_ptr (H * W * 3 floats of Welford sums) and frames_ptr (H * W uint32, or None), e.g. torch CUDA
        tensors' data_ptr().  Returns the AdaptiveResult."""
        if max_frames is None:
            max_frames = params.frames + 3 * (round_frames or params.frames)
        a = make_adaptive(target, max_frames, round_frames, floor)
        res = AdaptiveResult()
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_adaptive_device(self.h, scene.h, cam.ctypes.data, C.byref(params), C.byref(a),
                                                       C.c_void_p(out_ptr), C.c_void_p(m2_ptr),
                                                       C.c_void_p(frames_ptr) if frames_ptr else None, C.byref(res),
                                                       1 if sync else 0), "lt_render_adaptive_device")
        return res

    def debug_adaptive_part(self, parts, part):
        """Test hook: later adaptive calls render only the rows part `part` of a `parts`-device context would own
        (parts=1, part=0: the whole image again)"""
        self._check(self.lib.lt_debug_ctx_adaptive_part(self.h, parts, part), "lt_debug_ctx_adaptive_part")

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

    def render_plugin_cl(self, scene, camera, plugin_id, width, height, depth=3, kernel_mode=0, work_block=(0, 0),
                         group=(0, 0)):
        """An OpenCL C plug-in (a .cl file given to plugin_load), launched as the reference's OpenCL backend does: one
        launch per work block ((0, 0) = the whole image), work-group `group` ((0, 0) = the library's choice)."""
        out = np.zeros((height, width, depth), dtype=np.float32)
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_plugin_cl(self.h, scene.h, cam.ctypes.data, plugin_id, kernel_mode, width, height,
                                                 depth, work_block[0], work_block[1], group[0], group[1],
                                                 out.ctypes.data), "lt_render_plugin_cl")
        return out

    def render_plugin_frames(self, scene, camera, plugin_id, params, work_block=(0, 0), want_output=True):
        """params.frames frames of a plug-in combined by params.accum_mode (lt_render_plugin_frames), on one device or
        divided among the devices of a multi-device Context.  params.block_x/y: the CUDA block of a .cu plug-in, the
        work-group of a .cl plug-in; work_block: .cl plug-ins only.  Returns float32 [H, W, depth] or None."""
        out = np.empty((params.height, params.width, params.depth), dtype=np.float32) if want_output else None
        cam = np.ascontiguousarray(camera, dtype=L.CAMERA)
        self._check(self.lib.lt_render_plugin_frames(self.h, scene.h, cam.ctypes.data, plugin_id, C.byref(params),
                                                     work_block[0], work_block[1],
                                                     out.ctypes.data if out is not None else None),
                    "lt_render_plugin_frames")
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

    def uses_traversal_tree(self, scene):
        """Test hook: do the pruned threaded copies of `scene` walk a traversal tree (build_traversal_tree)?"""
        rc = self.lib.lt_debug_scene_traversal_tree(scene.h)
        self._check(min(rc, 0), "lt_debug_scene_traversal_tree")
        return rc == 1

    def scene_bytes(self, scene):
        """Test hook: the bytes of device memory `scene` holds (lt_debug_scene_bytes)"""
        out = C.c_uint64(0)
        self._check(self.lib.lt_debug_scene_bytes(scene.h, C.byref(out)), "lt_debug_scene_bytes")
        return out.value

    def debug_limits(self, threaded_max_nodes, stream_min_nodes):
        """Test hook: trees of at most threaded_max_nodes nodes get host-built threaded copies at upload (larger ones
        device-built copies); deterministic launches on scenes of at least stream_min_nodes nodes run k_flat_stream."""
        self._check(self.lib.lt_debug_ctx_limits(self.h, threaded_max_nodes, stream_min_nodes), "lt_debug_ctx_limits")

    def debug_list_order(self, reversed):
        """Test hook: later render_masked_device calls render their pixel list in reverse order (reversed=True) or in
        the compaction's order (False, the default); the output is the same either way."""
        self._check(self.lib.lt_debug_ctx_list_order(self.h, 1 if reversed else 0), "lt_debug_ctx_list_order")

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


def adaptive_rounds(params, aparams, first_frame_count=0):
    """Host-only: the frames of every round an adaptive call would render if every pixel kept going
    (lt_debug_adaptive_rounds), after the call's argument checks; raises LtError with the call's code and message."""
    lib = load()
    n = lib.lt_debug_adaptive_rounds(C.byref(params), C.byref(aparams) if aparams is not None else None,
                                     first_frame_count, None, 0)
    if n < 0:
        e = LtError("lt_render_adaptive failed (%d): %s" % (n, lib.lt_last_error(None).decode()))
        e.code = n
        raise e
    out = np.zeros(n, np.int32)
    lib.lt_debug_adaptive_rounds(C.byref(params), C.byref(aparams), first_frame_count, out.ctypes.data, n)
    return [int(x) for x in out]


PLAN_FIELDS = ("pipeline", "tree", "stats", "cull", "batch_frames", "streams", "rounds", "samples_per_frame",
               "shared_primary", "classify", "smem_stack", "smem_trace", "blocks_per_sm", "grid", "workspace_bytes")
PIPE_FLAT, PIPE_FLAT_STREAM, PIPE_PATH, PIPE_WAVEFRONT = range(4)
TREE_CHILD_PAIR, TREE_HOST_THREADED, TREE_DEVICE_THREADED = range(3)
ERR_INVALID, ERR_UNSUPPORTED = -1, -4


def plan(params, node_count, stack_depth, total_mem, sm_count):
    """Host-only: the launch plan lt_render makes for `params` on a scene of node_count nodes (lt_debug_plan), as a
    dict of PLAN_FIELDS plus "error" (0 or the code lt_render returns) and "message"."""
    lib = load()
    out = (C.c_int64 * len(PLAN_FIELDS))()
    rc = lib.lt_debug_plan(C.byref(params), node_count, stack_depth, total_mem, sm_count, out)
    if rc == ERR_INVALID:
        raise LtError("lt_debug_plan failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    d = dict(zip(PLAN_FIELDS, out))
    d["error"] = rc
    d["message"] = lib.lt_last_error(None).decode() if rc else ""
    return d


def plan_views(params, view_count, node_count, stack_depth, total_mem, sm_count):
    """Host-only: the launch plan of an lt_render_views call of view_count views (lt_debug_plan_views), as plan()."""
    lib = load()
    out = (C.c_int64 * len(PLAN_FIELDS))()
    rc = lib.lt_debug_plan_views(C.byref(params), view_count, node_count, stack_depth, total_mem, sm_count, out)
    if rc == ERR_INVALID:
        raise LtError("lt_debug_plan_views failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    d = dict(zip(PLAN_FIELDS, out))
    d["error"] = rc
    d["message"] = lib.lt_last_error(None).decode() if rc else ""
    return d


def plan_masked(params, pixel_count, node_count, stack_depth, total_mem, sm_count):
    """Host-only: the launch plan of an lt_render_masked_device call whose mask lists pixel_count pixels
    (lt_debug_plan_masked), as plan()."""
    lib = load()
    out = (C.c_int64 * len(PLAN_FIELDS))()
    rc = lib.lt_debug_plan_masked(C.byref(params), pixel_count, node_count, stack_depth, total_mem, sm_count, out)
    if rc == ERR_INVALID:
        raise LtError("lt_debug_plan_masked failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    d = dict(zip(PLAN_FIELDS, out))
    d["error"] = rc
    d["message"] = lib.lt_last_error(None).decode() if rc else ""
    return d


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


def build_traversal_tree(nodes, prim_count):
    """Host-only: the threaded records lt_scene_upload builds for a small tree (lt_debug_build_traversal_tree), as a
    dict: "full" (8 x N, the reference's copies), "pruned" (8 x stride; skip links index it flattened, like
    build_threaded_pruned), "stride", "traversal" (whether the pruned copies are a traversal tree over the reference's
    leaves rather than the reference tree) and "rank" (8 x prim_count, the equal-t tie-break table, or None)."""
    lib = load()
    nodes = np.ascontiguousarray(nodes)
    n = len(nodes)
    out = np.zeros(16 * n, THREAD_NODE)
    rank = np.zeros((8, prim_count), np.int32)
    stride, trav = C.c_int32(0), C.c_int32(0)
    rc = lib.lt_debug_build_traversal_tree(nodes.ctypes.data, nodes.nbytes, prim_count, out.ctypes.data,
                                           C.byref(stride), rank.ctypes.data, C.byref(trav))
    if rc != 0:
        raise LtError("lt_debug_build_traversal_tree failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    k = stride.value
    pruned = out[8 * n:8 * n + 8 * k].copy()
    pruned["skip"] = np.where(pruned["skip"] == -2147483648, pruned["skip"], pruned["skip"] - 8 * n)
    return {"full": out[:8 * n].reshape(8, n).copy(), "pruned": pruned.reshape(8, k), "stride": k,
            "traversal": trav.value == 1, "rank": rank if trav.value == 1 else None}


def traversal_tree(nodes, prim_count):
    """Host-only: the traversal tree lt_scene_upload builds for a small tree and the costs it is chosen by
    (lt_debug_traversal_tree), as a dict: "nodes" (the tree in the reference layout, or None when the tree gets none),
    "reference" (the expected box tests per root-hitting ray of the reference tree's pruned copies), "sah", "ploc" and
    "restructured" (those of the candidates over the reference's leaves, or None)."""
    lib = load()
    nodes = np.ascontiguousarray(nodes)
    out = np.zeros_like(nodes)
    cost = (C.c_double * 4)()
    rc = lib.lt_debug_traversal_tree(nodes.ctypes.data, nodes.nbytes, prim_count, out.ctypes.data, cost)
    if rc != 0:
        raise LtError("lt_debug_traversal_tree failed (%d): %s" % (rc, lib.lt_last_error(None).decode()))
    v = [None if np.isnan(x) else float(x) for x in cost]
    return {"nodes": None if v[1] is None else out, "reference": v[0], "sah": v[1], "ploc": v[2], "restructured": v[3]}

"""Shared helpers of the test-suite."""
import os

import numpy as np

from lens_trace_b200 import capi, host, layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = os.path.join(ROOT, "resources", "models")
GOLDEN = os.path.join(ROOT, "tests", "golden")

_cache = {}


def scene(name):
    """Flat buffers of resources/models/<name>.obj built by this repo's Model + AccelerationStructureExplicit."""
    if name not in _cache:
        _cache[name] = host.load_scene_buffers(os.path.join(MODELS, name + ".obj"))
    return _cache[name]


def default_camera(yaw=0.0, frame_count=0):
    # the camera every reference test and example uses (tests/cuda_renderer_test.cc:19)
    return L.make_camera(0, 2.5, -50, yaw, frame_count)


def device_group(n):
    """A multi-device Context of n members: devices 0 .. n-1 when torch sees that many, otherwise a shared group of n
    members on device 0 (capi.Context.shared), which runs every line of the multi-GPU code except the NCCL and peer
    mapping transport.  Use it in a `with` block, so that no member context or thread outlives the test."""
    import torch
    if torch.cuda.device_count() >= n:
        return capi.Context(list(range(n)))
    return capi.Context.shared(0, n)


def is_shared(ctx):
    """Whether a Context from device_group is a shared group (every member on one device)."""
    return ctx.shared_device is not None


def skip_nccl_without_two_gpus(exchange):
    """A test of the NCCL exchange needs a real group: a shared group's sample split always runs the p2p kernel, so on
    one GPU the nccl case would test that path a second time."""
    import pytest
    import torch
    if exchange == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("the nccl exchange needs two or more GPUs (a shared group combines with the p2p kernel)")


def group_sizes():
    """The member counts the multi-device tests use: every real device (up to 8) when there are two or more, and on
    one GPU 3 (not a power of two) and 8 (the largest count of a real group)."""
    import torch
    n = torch.cuda.device_count()
    return [min(n, 8)] if n >= 2 else [3, 8]


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_bit_equal(a, b, what=""):
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    bad = bits(a) != bits(b)
    if bad.any():
        idx = np.argwhere(bad)[:5]
        raise AssertionError("%s: %d of %d floats differ bitwise; first %s: %s vs %s" % (
            what, bad.sum(), bad.size, idx.tolist(), a[bad][:5], b[bad][:5]))


def single_triangle_scene(emissive=False):
    """A one-node tree (leaf root): exercises the root-leaf path."""
    nodes = np.zeros(1, L.NODE)
    nodes["min"][0] = (-1, 1.5, 0)
    nodes["max"][0] = (1, 3.5, 0)
    nodes["offset"][0] = 0
    nodes["count"][0] = 1
    prims = np.zeros(1, L.PRIM)
    prims["a"][0] = (-1, 1.5, 0)
    prims["b"][0] = (1, 1.5, 0)
    prims["c"][0] = (0, 3.5, 0)
    for k in ("na", "nb", "nc"):
        prims[k][0] = (0, 0, -1)
    mats = np.zeros(1, L.MATERIAL)
    mats["diffuse"][0] = (0.25, 0.5, 0.75)
    mats["ior"] = 1.0
    mats["dissolve"] = 1.0
    if emissive:
        mats["emission"][0] = (1, 1, 1)
    lights = np.zeros(1, L.LIGHTS)
    if emissive:
        lights["count"] = 1
    return L.SceneBuffers(nodes, prims, mats, lights)


def multi_prim_leaf_scene():
    """Reference-style buffers with a 2-primitive leaf (what the reference builder emits for
    coincident centroids): only the first primitive of the leaf may ever be hit (basic.cu:168-172)."""
    sb = scene("green_wall")
    nodes = np.zeros(1, L.NODE)
    nodes["min"][0] = sb.nodes["min"][0]
    nodes["max"][0] = sb.nodes["max"][0]
    nodes["offset"][0] = 0
    nodes["count"][0] = 2
    return L.SceneBuffers(nodes, sb.prims.copy(), sb.materials.copy(), sb.lights.copy())

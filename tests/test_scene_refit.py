"""lt_scene_refit without a device: a NumPy restatement of the refit, pinned against the host builder's boxes, and the
entry points' argument checks.

The restatement is the contract the GPU refit is compared with byte for byte (tests/test_gpu_scene_refit.py): a leaf's
box covers its primitiveCount primitives from primitivesOffset, in order; an inner node's box is the union of its first
child (i + 1) and its second (offset), in that order; min and max keep the first operand on ties, as std::min and
std::max do."""
import ctypes as C
import os

import numpy as np
import pytest

import util
from lens_trace_b200 import capi, host, layouts as L


def first_min(a, b):
    return np.where(b < a, b, a)


def first_max(a, b):
    return np.where(a < b, b, a)


def restate_refit(nodes, prims):
    """The node array lt_scene_refit leaves for `prims` on the topology of `nodes` (boxes of `nodes` are ignored)."""
    out = nodes.copy()
    n = len(out)
    count = out["count"].astype(np.int64)
    off = out["offset"].astype(np.int64)
    inner = np.nonzero(count == 0)[0]
    parent = np.full(n, -1, np.int64)
    parent[inner + 1] = inner
    parent[off[inner]] = inner
    depth = np.zeros(n, np.int64)
    for _ in range(n):  # parents precede their children in DFS order; one pass per level
        nd = np.where(parent >= 0, depth[np.maximum(parent, 0)] + 1, 0)
        if (nd == depth).all():
            break
        depth = nd
    lo = first_min(first_min(prims["a"], prims["b"]), prims["c"])
    hi = first_max(first_max(prims["a"], prims["b"]), prims["c"])
    leaf = np.nonzero(count > 0)[0]
    mn, mx = lo[off[leaf]], hi[off[leaf]]
    for j in range(1, int(count.max()) if len(leaf) else 1):
        more = count[leaf] > j
        idx = off[leaf[more]] + j
        mn[more] = first_min(mn[more], lo[idx])
        mx[more] = first_max(mx[more], hi[idx])
    out["min"][leaf], out["max"][leaf] = mn, mx
    for d in range(int(depth.max()), -1, -1):
        level = inner[depth[inner] == d]
        a, b = level + 1, off[level]
        out["min"][level] = first_min(out["min"][a], out["min"][b])
        out["max"][level] = first_max(out["max"][a], out["max"][b])
    return out


def zero_boxes(nodes):
    z = nodes.copy()
    z["min"] = 0
    z["max"] = 0
    return z


def positive_zeros(nodes):
    z = nodes.copy()
    z["min"] += np.float32(0)  # -0 + 0 = +0
    z["max"] += np.float32(0)
    return z


# Signed zeros inside triangles: the bounds of each triangle depend on the operand order (std::min(+0, -0) is +0,
# std::max(-0, +0) is -0), and each zero bound is the extreme of the whole scene on its axis for one triangle only.
SIGNED_ZERO_OBJ = """v 0 0.5 1
v -0 1 2
v 1 1.5 3
v 2 -0 4
v 3 0 5
v 2.5 -1 6
v 4 2 -0
v 5 3 0
v 4.5 2.5 -1
v -1 -2 7
v -0.5 -3 8
v -0 -2.5 9
f 1 2 3
f 4 5 6
f 7 8 9
f 10 11 12
"""


@pytest.fixture(scope="module")
def signed_zero_scene(tmp_path_factory):
    path = os.path.join(str(tmp_path_factory.mktemp("refit")), "signed_zero.obj")
    with open(path, "w") as f:
        f.write(SIGNED_ZERO_OBJ)
    return host.load_scene_buffers(path)


@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens"])
def test_restatement_reproduces_host_builder(name):
    sb = util.scene(name)
    got = restate_refit(zero_boxes(sb.nodes), sb.prims)
    # The builder folds an inner node's box over its primitives in its partition order, which the tree does not
    # record, so of -0 and +0 its inner boxes may keep the other one (Cornell box root: min y +0, refit -0).  The
    # values are equal; every other bit is the builder's.
    assert positive_zeros(got).tobytes() == positive_zeros(sb.nodes).tobytes()
    leaf = sb.nodes["count"] > 0
    assert got[leaf].tobytes() == sb.nodes[leaf].tobytes()


def test_restatement_multi_primitive_leaf():
    sb = util.multi_prim_leaf_scene()
    got = restate_refit(zero_boxes(sb.nodes), sb.prims)
    assert got.tobytes() == sb.nodes.tobytes()
    # the box covers both primitives, not only the first one the reference's leaf tests
    moved = sb.prims.copy()
    for k in ("a", "b", "c"):
        moved[k][1] += np.float32(10)
    assert (restate_refit(sb.nodes, moved)["max"][0] > got["max"][0]).all()


def test_restatement_signed_zeros(signed_zero_scene):
    sb = signed_zero_scene
    assert np.signbit(sb.prims["a"]).any() or np.signbit(sb.prims["b"]).any()
    got = restate_refit(zero_boxes(sb.nodes), sb.prims)
    assert got.tobytes() == sb.nodes.tobytes()
    # both signs of zero are bounds, each taken from a triangle that holds the other sign too
    zmin = sb.nodes["min"][sb.nodes["min"] == 0]
    zmax = sb.nodes["max"][sb.nodes["max"] == 0]
    assert (~np.signbit(zmin)).any() and np.signbit(zmax).any()


def test_restatement_is_the_union_of_children():
    sb = util.scene("cornell_box_lens")
    rng = np.random.default_rng(7)
    prims = sb.prims.copy()
    for k in ("a", "b", "c"):
        prims[k] += rng.normal(scale=0.05, size=prims[k].shape).astype(np.float32)
    got = restate_refit(sb.nodes, prims)
    for i in np.nonzero(got["count"] == 0)[0]:
        a, b = got[i + 1], got[got["offset"][i]]
        assert (got["min"][i] == np.minimum(a["min"], b["min"])).all()
        assert (got["max"][i] == np.maximum(a["max"], b["max"])).all()
    assert (got["offset"] == sb.nodes["offset"]).all() and (got["axis"] == sb.nodes["axis"]).all()


def test_entry_points_exist():
    lib = capi.load()
    for s in ("lt_scene_refit", "lt_scene_refit_device"):
        assert hasattr(lib, s) and s in capi.SYMBOLS
    assert hasattr(capi.Context, "refit") and hasattr(capi.Context, "refit_device")


@pytest.mark.parametrize("entry", ["lt_scene_refit", "lt_scene_refit_device"])
def test_null_ctx_without_a_device(entry):
    lib = capi.load()
    fn = getattr(lib, entry)
    prims = np.zeros(2, L.PRIM)
    for scene, buf in ((None, None), (None, prims.ctypes.data), (C.c_void_p(0x1000), None),
                       (C.c_void_p(0x1000), prims.ctypes.data)):
        assert fn(None, scene, buf, prims.nbytes) == capi.ERR_INVALID
        assert b"ctx is NULL" in lib.lt_last_error(None)

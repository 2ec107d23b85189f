"""lt_scene_build_ploc: the PLOC tree built on the device (lens_trace_b200/csrc/lt_bvh.cu), against a NumPy
restatement of the same algorithm -- Morton keys, search radius, float32 half-area order, tie key, id allocation and
emission -- which must give the same bytes.  The CPU tests check the restatement's trees; the GPU tests check the
device against it, and the kernels against the oracle on the device's trees."""
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L
from test_host import _check_tree
from test_threaded_prune import _check_same_leaves

PLOC_RADIUS = 8  # lt_bvh.cu
f32 = np.float32
M32 = 0xFFFFFFFF


# ---- the restatement ----

def _fmin(a, b):
    """fminf / fmaxf on the device: -0 is below +0"""
    return np.where(a == b, np.where(np.signbit(a), a, b), np.minimum(a, b))


def _fmax(a, b):
    return np.where(a == b, np.where(np.signbit(a), b, a), np.maximum(a, b))


def _prim_boxes(prims):
    lo = _fmin(_fmin(prims["a"], prims["b"]), prims["c"]).astype(f32)
    hi = _fmax(_fmax(prims["a"], prims["b"]), prims["c"]).astype(f32)
    return lo, hi


def _spread21(v):
    x = v.astype(np.uint64) & np.uint64(0x1FFFFF)
    for shift, mask in ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F),
                        (4, 0x10C30C30C30C30C3), (2, 0x1249249249249249)):
        x = (x | (x << np.uint64(shift))) & np.uint64(mask)
    return x


def _morton_order(lo, hi):
    """k_centroid_bounds, k_morton and the stable radix sort: leaf position -> input index."""
    c = f32(0.5) * lo + f32(0.5) * hi
    mn, mx = c.min(axis=0), c.max(axis=0)
    ext = mx - mn
    with np.errstate(all="ignore"):
        u = np.where(ext > 0, (c - mn) / np.where(ext > 0, ext, f32(1)), f32(0)).astype(f32)
    q = np.minimum(np.maximum(u * f32(2097152.0), f32(0)), f32(2097151.0)).astype(np.uint32)
    key = (_spread21(q[:, 0]) << np.uint64(2)) | (_spread21(q[:, 1]) << np.uint64(1)) | _spread21(q[:, 2])
    return np.argsort(key, kind="stable")


def _pair_hash(a, b):
    h = (a.astype(np.uint64) ^ ((b.astype(np.uint64) * 0x9E3779B9) & M32)) & M32
    h ^= h >> np.uint64(16)
    h = (h * 0x85EBCA6B) & M32
    h ^= h >> np.uint64(13)
    h = (h * 0xC2B2AE35) & M32
    h ^= h >> np.uint64(16)
    return h


def _nearest(lo, hi):
    """k_ploc_nn: per position the neighbour within PLOC_RADIUS with the smallest (half-area bits, hash, min, max)."""
    m = len(lo)
    i = np.arange(m)
    bd = np.zeros(m, np.uint64)
    bh = np.zeros(m, np.uint64)
    ba = np.zeros(m, np.int64)
    bb = np.zeros(m, np.int64)
    best = np.full(m, -1, np.int64)
    for o in range(-PLOC_RADIUS, PLOC_RADIUS + 1):
        j = i + o
        ok = (o != 0) & (j >= 0) & (j < m)
        jj = np.clip(j, 0, m - 1)
        e = _fmax(hi, hi[jj]) - _fmin(lo, lo[jj])
        area = (e[:, 0] * e[:, 1] + e[:, 1] * e[:, 2]) + e[:, 2] * e[:, 0]
        d = area.astype(f32).view(np.uint32).astype(np.uint64)
        a, b = np.minimum(i, j), np.maximum(i, j)
        h = _pair_hash(a, b)
        better = ok & ((best < 0) | (d < bd) | ((d == bd) & ((h < bh) | ((h == bh) & ((a < ba) | ((a == ba) & (b < bb)))))))
        best = np.where(better, j, best)
        bd, bh, ba, bb = (np.where(better, x, y) for x, y in ((d, bd), (h, bh), (a, ba), (b, bb)))
    assert (best >= 0).all()
    return best


class Tree:
    """children (n-1, 2) with leaves as ~position, inner boxes, axes, leaf order (position -> input index)"""

    def __init__(self, n):
        self.children = np.zeros((n - 1, 2), np.int64)
        self.lo = np.zeros((n - 1, 3), f32)
        self.hi = np.zeros((n - 1, 3), f32)
        self.axis = np.zeros(n - 1, np.int64)
        self.leaves = np.zeros(n - 1, np.int64)
        self.iterations = 0


def ploc_tree(prims):
    lo, hi = _prim_boxes(prims)
    n = len(prims)
    order = _morton_order(lo, hi)
    T = Tree(n)
    T.order = order
    node = ~np.arange(n, dtype=np.int64)
    clo, chi = lo[order], hi[order]
    m = n
    while m > 1:
        nn = _nearest(clo, chi)
        i = np.arange(m)
        mutual = nn[nn] == i
        merge = mutual & (i < nn)
        keep = ~(mutual & (nn < i))
        rank = np.cumsum(merge) - merge
        pos = np.cumsum(keep) - keep
        A = i[merge]
        B = nn[A]
        ids = m - 2 - rank[A]
        ca = f32(0.5) * clo[A] + f32(0.5) * chi[A]
        cb = f32(0.5) * clo[B] + f32(0.5) * chi[B]
        ax = np.argmax(np.abs(ca - cb), axis=1)
        r = np.arange(len(A))
        swap = cb[r, ax] < ca[r, ax]
        first = np.where(swap, node[B], node[A])
        second = np.where(swap, node[A], node[B])
        ulo, uhi = _fmin(clo[A], clo[B]), _fmax(chi[A], chi[B])
        T.children[ids, 0], T.children[ids, 1] = first, second
        T.lo[ids], T.hi[ids], T.axis[ids] = ulo, uhi, ax
        lf = lambda v: np.where(v < 0, 1, T.leaves[np.maximum(v, 0)])
        T.leaves[ids] = lf(first) + lf(second)
        nxt = int(keep.sum())
        assert nxt < m
        nnode = np.empty(nxt, np.int64)
        nlo, nhi = np.empty((nxt, 3), f32), np.empty((nxt, 3), f32)
        nnode[pos[keep]], nlo[pos[keep]], nhi[pos[keep]] = node[keep], clo[keep], chi[keep]
        nnode[pos[A]], nlo[pos[A]], nhi[pos[A]] = ids, ulo, uhi
        node, clo, chi, m = nnode, nlo, nhi, nxt
        T.iterations += 1
    assert node[0] == 0
    return T


def emit(T, prims, materials):
    """k_dfs_index / k_emit_nodes / the light selection: (SceneBuffers, stack depth)"""
    n = len(prims)
    lo, hi = _prim_boxes(prims)
    nodes = np.zeros(2 * n - 1, L.NODE)
    ordered = np.zeros(n, L.PRIM)
    slot, leaf_rank, depth = 0, 0, 0
    stack = [(0, 0, None)]  # (reference, inner ancestors, parent slot to patch with the DFS index)
    while stack:
        ref, d, patch = stack.pop()
        if patch is not None:
            nodes["offset"][patch] = slot
        if ref < 0:
            src = T.order[~ref]
            ordered[leaf_rank] = prims[src]
            nodes["min"][slot], nodes["max"][slot] = lo[src], hi[src]
            nodes["offset"][slot], nodes["count"][slot] = leaf_rank, 1
            leaf_rank += 1
            depth = max(depth, d)
        else:
            nodes["min"][slot], nodes["max"][slot], nodes["axis"][slot] = T.lo[ref], T.hi[ref], T.axis[ref]
            stack.append((int(T.children[ref, 1]), d + 1, slot))
            stack.append((int(T.children[ref, 0]), d + 1, None))
        slot += 1
    lights = np.zeros(1, L.LIGHTS)
    emissive = np.nonzero((materials["emission"][ordered["mat"]] > 0).any(axis=1))[0][:64]
    lights["count"][0] = len(emissive)
    lights["prims"][0][:len(emissive)] = emissive
    return L.SceneBuffers(nodes, ordered, materials, lights), depth


def sah_cost(nodes):
    inner = nodes[nodes["count"] == 0]
    e = (inner["max"] - inner["min"]).astype(np.float64)
    r = (nodes["max"][0] - nodes["min"][0]).astype(np.float64)
    half = lambda x: x[..., 0] * x[..., 1] + x[..., 1] * x[..., 2] + x[..., 2] * x[..., 0]
    return half(e).sum() / half(r)


# ---- inputs ----

def _write_obj(path, tris, emissive_last=False):
    base = os.path.splitext(path)[0]
    with open(base + ".mtl", "w") as f:
        f.write("newmtl M\nKd 0.5 0.5 0.5\nnewmtl E\nKd 1 1 1\nKe 4 4 4\n")
    with open(path, "w") as f:
        f.write("mtllib %s.mtl\nusemtl M\n" % os.path.basename(base))
        for k, t in enumerate(tris):
            if emissive_last and k == len(tris) - 1:
                f.write("usemtl E\n")
            for v in t:
                f.write("v %r %r %r\n" % tuple(float(x) for x in v))
            f.write("f %d %d %d\n" % (3 * k + 1, 3 * k + 2, 3 * k + 3))


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    """name -> OBJ path: the shipped models, a small synthetic mesh, 1 000 copies of one triangle, two triangles"""
    d = tmp_path_factory.mktemp("ploc")
    paths = {name: os.path.join(util.MODELS, name + ".obj") for name in ("green_wall", "cornell_box", "cornell_box_lens")}
    paths["synthetic"] = str(d / "synthetic.obj")
    host.write_synthetic_scene(paths["synthetic"], 10, 0x5EED)
    paths["coincident"] = str(d / "coincident.obj")
    _write_obj(paths["coincident"], [((0, 0, 0), (1, 0, 0), (0, 1, 0))] * 1000)
    paths["two"] = str(d / "two.obj")
    _write_obj(paths["two"], [((0, 0, 0), (1, 0, 0), (0, 1, 0)), ((3, 1, 2), (4, 2, 2), (3, 3, 5))], emissive_last=True)
    return paths


INPUTS = ["green_wall", "cornell_box", "cornell_box_lens", "synthetic", "coincident", "two"]
_median = {}


def _load(path):
    """(primitives in a fixed shuffled order, materials, median-split buffers)"""
    if path not in _median:
        sb = host.load_scene_buffers(path)
        perm = np.random.default_rng(5).permutation(len(sb.prims))
        _median[path] = (sb.prims[perm].copy(), sb.materials.copy(), sb)
    return _median[path]


def reference(path):
    prims, mats, median = _load(path)
    T = ploc_tree(prims)
    sb, depth = emit(T, prims, mats)
    return prims, mats, median, sb, depth, T


# ---- CPU: the restatement's trees ----

@pytest.mark.parametrize("name", INPUTS)
def test_restated_tree_is_valid_and_no_worse_than_the_median_split(inputs, name):
    prims, mats, median, sb, depth, _ = reference(inputs[name])
    _check_tree(sb)
    assert sorted(p.tobytes() for p in sb.prims) == sorted(p.tobytes() for p in prims)
    assert sb.lights["count"][0] == median.lights["count"][0]
    assert 1 <= depth <= 64
    capi.build_threaded(sb.nodes)  # passes the upload-time validation
    assert sah_cost(sb.nodes) <= sah_cost(median.nodes)
    _check_same_leaves(sb.nodes, np.random.default_rng(11), n_rays=1500)


def test_coincident_triangles_give_a_shallow_tree(inputs):
    """With the mixed tie key many pairs merge per iteration even when every area is equal (the rule "smaller
    neighbour on equal area" would merge one pair per iteration and build a chain)."""
    _, _, _, _, depth, T = reference(inputs["coincident"])
    assert depth == COINCIDENT_DEPTH <= 32
    assert T.iterations <= 32


COINCIDENT_DEPTH = 18


def test_without_a_device_the_ploc_option_builds_the_host_sah_tree(inputs):
    try:
        c = capi.Context(0)
    except capi.LtError:
        c = None
    if c is not None:
        c.close()
        pytest.skip("a CUDA device is usable")
    for name in ("cornell_box", "synthetic"):
        a = host.load_scene_buffers(inputs[name], host.AccelerationStructure.GPU_PLOC)
        b = host.load_scene_buffers(inputs[name], host.AccelerationStructure.HOST_SAH)
        assert a.nodes.tobytes() == b.nodes.tobytes() and a.prims.tobytes() == b.prims.tobytes()
        assert a.lights.tobytes() == b.lights.tobytes()


# ---- GPU ----

@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def large(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("ploc_large") / "synth.obj")
    host.write_synthetic_scene(p, 200, 0x5EED)  # 80 012 triangles (exercises the parallel light selection)
    return p


def _assert_same_bytes(got, depth, want, want_depth):
    assert got.nodes.tobytes() == want.nodes.tobytes(), np.nonzero(got.nodes != want.nodes)[0][:5]
    assert got.prims.tobytes() == want.prims.tobytes()
    assert got.lights.tobytes() == want.lights.tobytes()
    assert depth == want_depth


@pytest.mark.gpu
@pytest.mark.parametrize("name", INPUTS + ["large"])
def test_device_tree_equals_the_restatement(ctx, inputs, large, name):
    path = large if name == "large" else inputs[name]
    prims, mats, median, want, want_depth, _ = reference(path)
    sc = ctx.build_ploc(prims, mats)
    got, depth = ctx.download(sc)
    _assert_same_bytes(got, depth, want, want_depth)
    again = ctx.build_ploc(prims, mats)
    _assert_same_bytes(ctx.download(again)[0], ctx.download(again)[1], want, want_depth)
    _check_tree(got)
    assert got.lights["count"][0] == median.lights["count"][0]
    sc.release()
    again.release()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "green_wall"])
def test_kernels_equal_the_oracle_on_the_ploc_tree(ctx, name):
    from test_gpu_parity import assert_images_match
    prims, mats, median = _load(os.path.join(util.MODELS, name + ".obj"))
    sc = ctx.build_ploc(prims, mats)
    sb, depth = ctx.download(sc)
    _check_tree(sb)
    assert sorted(p.tobytes() for p in sb.prims) == sorted(p.tobytes() for p in prims)
    n = sb.lights["count"][0]
    assert n == median.lights["count"][0]
    cam = util.default_camera(0.03, 1)
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, 200, 150)
    oids, ohit, otuv, _ = O.primary_hits(0, sb, cam, 200, 150)
    np.testing.assert_array_equal(hit, ohit)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv, "PLOC: kernels vs oracle on the same buffers")
    want = O.render(L.KERNEL_GI, sb, cam, 160, 120, max_ray_depth=4, threads=0)
    for flags in (L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT):
        got = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 160, 120, max_ray_depth=4, flags=flags))
        assert_images_match(got, want, "PLOC GI (flags %d) vs oracle" % flags, max_outliers=3)
    _check_same_leaves(sb.nodes, np.random.default_rng(3))
    sc.release()


@pytest.mark.gpu
def test_large_mesh_against_the_oracle_and_the_lbvh(ctx, large):
    prims, mats, median = _load(large)
    sc = ctx.build_ploc(prims, mats)
    sb, depth = ctx.download(sc)
    _check_tree(sb)
    assert sb.lights["count"][0] == median.lights["count"][0] == 2 and depth <= 64
    cam = util.default_camera()
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 320, 180)
    oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, 320, 180)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv)
    lb = ctx.build_lbvh(prims, mats)
    lsb, _ = ctx.download(lb)
    assert sah_cost(sb.nodes) <= sah_cost(lsb.nodes)

    def box_tests(scene):
        p = capi.make_params(L.KERNEL_GI, 320, 180, max_ray_depth=4, flags=L.FLAG_STATS)
        ctx.render(scene, cam, p, want_output=False)
        s = ctx.stats()
        return s.node_tests / s.rays

    assert box_tests(sc) <= box_tests(lb)
    lb.release()
    sc.release()


@pytest.mark.gpu
def test_acceleration_structure_gpu_ploc_option():
    """AccelerationStructureExplicit with ACCELERATION_STRUCTURE_TYPE_PLOC_B200: built on the GPU, held on the host
    in the reference layout, rendered through RendererCUDA bit-equal to the oracle on its own buffers."""
    os.chdir(util.ROOT)
    cam = host.Camera(0, 2.5, -50, 0)
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model, host.AccelerationStructure.GPU_PLOC)
    sb = accel.buffers()
    assert len(sb.nodes) == 83 and sb.lights["count"][0] == 2
    _check_tree(sb)
    sah = host.load_scene_buffers("resources/models/cornell_box.obj", host.AccelerationStructure.HOST_SAH)
    assert sb.nodes.tobytes() != sah.nodes.tobytes()  # the device tree, not the host fallback
    r = host.Renderer(host.PLATFORM_CUDA)
    got = r.render("resources/kernels/cuda/basic.cu", 128, 96, accel, model, cam)
    util.assert_bit_equal(got, O.render(L.KERNEL_BASIC_CU, sb, util.default_camera(), 128, 96))
    r.close(); accel.close(); model.close(); cam.close()


def _rc(c, prims, mats):
    out = capi.C.c_void_p()
    rc = c.lib.lt_scene_build_ploc(c.h, prims.ctypes.data, prims.nbytes, mats.ctypes.data, mats.nbytes,
                                   capi.C.byref(out))
    if rc == 0:
        c.lib.lt_scene_release(c.h, out)
    return rc


@pytest.mark.gpu
def test_error_cases(ctx):
    prims, mats, _ = _load(os.path.join(util.MODELS, "cornell_box.obj"))
    assert _rc(ctx, prims, mats) == 0
    assert _rc(ctx, prims[:1].copy(), mats) == -4  # fewer than two primitives: LT_ERR_UNSUPPORTED
    raw = np.frombuffer(prims.tobytes() + b"\0", np.uint8)
    out = capi.C.c_void_p()
    assert ctx.lib.lt_scene_build_ploc(ctx.h, raw.ctypes.data, raw.nbytes, mats.ctypes.data, mats.nbytes,
                                       capi.C.byref(out)) == -1  # not a multiple of the record size
    bad = prims.copy()
    bad["mat"][3] = len(mats)
    assert _rc(ctx, bad, mats) == -1  # materialIndex out of range
    for v in (np.inf, -np.inf, np.nan):
        bad = prims.copy()
        bad["b"][7, 1] = v
        assert _rc(ctx, bad, mats) == -1  # non-finite vertex
        assert "non-finite" in ctx.lib.lt_last_error(ctx.h).decode()
    with pytest.raises(capi.LtError):
        ctx.build_ploc(prims[:1], mats)


@pytest.mark.gpu
def test_multi_gpu_context_is_refused():
    prims, mats, _ = _load(os.path.join(util.MODELS, "cornell_box.obj"))
    c = util.device_group(2)
    assert _rc(c, prims, mats) == -4
    assert "single-GPU context" in c.lib.lt_last_error(c.h).decode()
    c.close()

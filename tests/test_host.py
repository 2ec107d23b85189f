"""CPU tests of the host surface: OBJ loader, BVH builder, scene parser, kernel-path registry, and the
C-ABI libraries' exported symbols (no compute without a GPU)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L


def test_libraries_export_every_declared_symbol():
    lib = capi.load()
    for name in capi.SYMBOLS:
        assert hasattr(lib, name), name
    hl = host.load()
    for name in host.SYMBOLS:
        assert hasattr(hl, name), name
    assert lib.lt_api_version() == 2
    # every function the header declares is bound above
    header = open(os.path.join(util.ROOT, "include", "lens_trace_b200.h")).read()
    import re
    declared = set(re.findall(r"\b(lt_[a-z_]+)\s*\(", header))
    assert declared == set(capi.SYMBOLS), declared ^ set(capi.SYMBOLS)


def test_no_silent_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(capi.LtError) as e:
        capi.Context(0)
    assert "no CUDA device" in str(e.value) and "no CPU fallback" in str(e.value)


def test_kernel_registry(tmp_path):
    """kernelFilePath -> pipeline goes by the file's content, never by its name (renderer_cuda.cpp:20-39,52-55
    compiles whatever the file holds)."""
    k = capi.kernel_from_path
    R = util.ROOT
    assert k(os.path.join(R, "resources/kernels/cuda/basic.cu")) == L.KERNEL_BASIC_CU
    assert k(os.path.join(R, "resources/kernels/opencl/basic.cl")) == L.KERNEL_BASIC_CL
    assert k(os.path.join(R, "examples/custom_kernel/resources/kernels/custom_opencl.cl")) == L.KERNEL_CUSTOM_BARY
    assert k(os.path.join(R, "resources/kernels/opencl/basic_lighting.cl")) == L.KERNEL_LIGHTING25
    assert k(os.path.join(R, "examples/accumulator/resources/kernels/accumulator.cl")) == L.KERNEL_ACCUMULATOR
    assert k(os.path.join(R, "resources/kernels/opencl/global_illumination.cl")) == L.KERNEL_GI25
    assert k(os.path.join(R, "examples/global_illumination/resources/kernels/global_illumination.cl")) == L.KERNEL_GI
    assert k("/nonexistent/resources/kernels/cuda/basic.cu") < 0  # unreadable: nothing to go by
    assert k("my_own_kernel.cl") < 0
    # a descriptor under any name selects its pipeline; the same name with other content does not
    d = tmp_path / "whatever.cl"
    d.write_text("// my scene\n// lt-pipeline: gi25\n")
    assert k(str(d)) == L.KERNEL_GI25
    edited = tmp_path / "basic.cu"
    edited.write_text(open(os.path.join(R, "resources/kernels/cuda/basic.cu")).read() +
                      'extern "C" __global__ void linearKernel() {}\n')
    assert k(str(edited)) < 0  # descriptor tag + code = a user kernel
    cl = tmp_path / "custom_opencl.cl"
    cl.write_text("__kernel void linearKernel() {}\n")
    assert k(str(cl)) < 0


REF_KERNELS = [("resources/kernels/cuda/basic.cu", L.KERNEL_BASIC_CU),
               ("resources/kernels/opencl/basic.cl", L.KERNEL_BASIC_CL),
               ("examples/custom_kernel/resources/kernels/custom_opencl.cl", L.KERNEL_CUSTOM_BARY),
               ("resources/kernels/opencl/basic_lighting.cl", L.KERNEL_LIGHTING25),
               ("examples/accumulator/resources/kernels/accumulator.cl", L.KERNEL_ACCUMULATOR),
               ("resources/kernels/opencl/global_illumination.cl", L.KERNEL_GI25),
               ("examples/global_illumination/resources/kernels/global_illumination.cl", L.KERNEL_GI)]


@pytest.mark.skipif(not os.path.isdir("/root/reference"), reason="the reference tree is only present in the build container")
def test_kernel_registry_recognises_the_reference_text(tmp_path):
    """The reference's own kernel files (unmodified, also with CRLF line ends, under any name) select the built-in
    pipeline; one changed character makes the file a user kernel."""
    k = capi.kernel_from_path
    for rel, kernel in REF_KERNELS:
        src = os.path.join("/root/reference", rel)
        assert k(src) == kernel, rel
        text = open(src, "rb").read()
        crlf = tmp_path / ("crlf_" + os.path.basename(rel))
        crlf.write_bytes(text.replace(b"\n", b"\r\n"))
        assert k(str(crlf)) == kernel
        edited = tmp_path / os.path.basename(rel)
        edited.write_bytes(text.replace(b"0.5", b"0.4", 1) if b"0.5" in text else text + b"\n// x\n")
        assert k(str(edited)) < 0, rel


def test_cornell_box_loads_like_the_reference():
    sb = util.scene("cornell_box")
    assert len(sb.prims) == 42 and len(sb.nodes) == 83 and len(sb.materials) == 5
    assert sb.lights["count"][0] == 2
    lens = util.scene("cornell_box_lens")
    assert len(lens.prims) == 166 and len(lens.nodes) == 331 and len(lens.materials) == 6
    assert (lens.materials["dissolve"] < 1).sum() == 1  # Material.005, d 0.25
    # light primitives are the emissive ones
    for sbx in (sb, lens):
        n = sbx.lights["count"][0]
        for p in sbx.lights["prims"][0][:n]:
            assert sbx.materials["emission"][sbx.prims["mat"][p]].max() > 0


@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens"])
def test_model_loader_matches_the_reference_loader_golden(name):
    """This repo's OBJ/MTL reader on resources/models vs the triangles and materials the reference's loader made
    (stored in tests/golden/ref_cuda_*.npz): the same primitives, in the reference builder's order or not."""
    z = np.load(os.path.join(util.GOLDEN, "ref_cuda_%s_yaw000.npz" % name))
    sb = util.scene(name)
    key = lambda p: p.tobytes()
    assert sorted(map(key, sb.prims)) == sorted(map(key, z["prims"]))
    assert sb.materials.tobytes() == z["materials"].tobytes()


def test_quad_split_rule(tmp_path):
    # shorter diagonal; a tie takes [0,1,3],[1,2,3] (tiny_obj_loader.h:1447-1487)
    obj = tmp_path / "q.obj"
    (tmp_path / "q.mtl").write_text("newmtl M\nKd 1 1 1\n")
    obj.write_text("mtllib q.mtl\nusemtl M\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nv 0 0 1\nv 4 0 1\nv 5 1 1\nv 0 1 1\n"
                   "vn 0 0 1\nf 1//1 2//1 3//1 4//1\nf -4//1 -3//1 -2//1 -1//1\n")
    m = host.Model(str(obj))
    assert m.primitive_count == 4
    a = host.AccelerationStructure(m)
    sb = a.buffers()
    tris = {tuple(map(tuple, np.stack([p["a"], p["b"], p["c"]]).tolist())) for p in sb.prims}
    assert ((0, 0, 0), (1, 0, 0), (0, 1, 0)) in tris and ((1, 0, 0), (1, 1, 0), (0, 1, 0)) in tris  # tie
    # second quad: diagonal 0-2 is (5,1) long, 1-3 is (4,1): 1-3 shorter -> [0,1,3],[1,2,3]
    assert ((0, 0, 1), (4, 0, 1), (0, 1, 1)) in tris and ((4, 0, 1), (5, 1, 1), (0, 1, 1)) in tris
    a.close()
    m.close()


def _check_tree(sb):
    nodes, n = sb.nodes, len(sb.nodes)
    seen = np.zeros(len(sb.prims), int)

    def walk(i):
        nd = nodes[i]
        if nd["count"] > 0:
            assert nd["count"] == 1
            p = sb.prims[nd["offset"]]
            pts = np.stack([p["a"], p["b"], p["c"]])
            np.testing.assert_array_equal(nd["min"], pts.min(0))
            np.testing.assert_array_equal(nd["max"], pts.max(0))
            seen[nd["offset"]] += 1
            return nd["min"], nd["max"], i + 1
        lmin, lmax, nxt = walk(i + 1)
        assert nd["offset"] == nxt  # DFS order: second child follows the first subtree
        rmin, rmax, nxt = walk(nd["offset"])
        np.testing.assert_array_equal(nd["min"], np.minimum(lmin, rmin))
        np.testing.assert_array_equal(nd["max"], np.maximum(lmax, rmax))
        assert nd["axis"] in (0, 1, 2)
        return nd["min"], nd["max"], nxt

    _, _, end = walk(0)
    assert end == n and (seen == 1).all()


def test_bvh_invariants():
    for name in ("green_wall", "cornell_box", "cornell_box_lens"):
        _check_tree(util.scene(name))


def test_builder_is_deterministic():
    a = host.load_scene_buffers(os.path.join(util.MODELS, "cornell_box_lens.obj"))
    b = host.load_scene_buffers(os.path.join(util.MODELS, "cornell_box_lens.obj"))
    assert a.nodes.tobytes() == b.nodes.tobytes() and a.prims.tobytes() == b.prims.tobytes()
    assert a.lights.tobytes() == b.lights.tobytes()


def test_synthetic_scene(tmp_path):
    p = str(tmp_path / "s.obj")
    n = host.write_synthetic_scene(p, 24, 0x5EED)
    assert n == 12 + 2 * 24 * 24
    sb = host.load_scene_buffers(p)
    assert len(sb.prims) == n and len(sb.nodes) == 2 * n - 1
    assert sb.lights["count"][0] == 2
    _check_tree(sb)
    q = str(tmp_path / "t.obj")
    host.write_synthetic_scene(q, 24, 0x5EED)
    assert open(p).read().split("\n", 1)[1] == open(q).read().split("\n", 1)[1].replace("t.mtl", "s.mtl")
    assert sb.prims["min" if False else "a"].min() >= -2.5001 and sb.prims["a"][:, 1].max() <= 5.0001


def test_camera_buffer_layout():
    c = host.Camera(1, 2, 3, 0.5)
    b = c.buffer()
    assert tuple(b["pos"][0]) == (1, 2, 3) and b["yaw"][0] == np.float32(0.5) and b["frameCount"][0] == 0
    c.increment_frame_count()
    c.increment_frame_count()
    assert c.buffer()["frameCount"][0] == 2
    c.set_frame_count(0)
    assert c.buffer()["frameCount"][0] == 0
    c.close()


def test_scene_files_parse(tmp_path):
    # run_scene_file needs a GPU to render; here only the parser: a bad file is reported, not fatal
    bad = tmp_path / "bad.scene"
    bad.write_text("{ not json")
    out = np.zeros(4, np.float32)
    dims = (C.c_uint64 * 3)()
    rc = host.load().lth_run_scene_file(str(bad).encode(), out.ctypes.data, out.nbytes, C.byref(dims))
    assert rc == -1
    for f in os.listdir(os.path.join(util.ROOT, "resources", "scenes")):
        json.load(open(os.path.join(util.ROOT, "resources", "scenes", f)))


def test_reference_sources_compile_against_these_headers(tmp_path):
    """Drop-in at the source level: the reference's own example and CLI compile, unedited, against
    include/lens_trace (needs /root/reference; skipped on the GPU box)."""
    import subprocess
    ref = "/root/reference"
    if not os.path.isdir(ref):
        pytest.skip("reference sources not present")
    inc = os.path.join(util.ROOT, "include")
    for src, defs in ((ref + "/examples/custom_kernel/src/main.cpp", []),
                      (ref + "/src/main.cpp", ["-DCUDA_ENABLED", "-DOPENCL_ENABLED"])):
        r = subprocess.run(["/usr/bin/g++", "-fsyntax-only", "-I", inc] + defs + [src], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr


def _slab(lo, hi, o, inv):
    """intersectBounds (basic.cu:136-154) on dirIsNeg-selected bounds, FP32, NaN semantics of the select chain"""
    f = np.float32
    with np.errstate(all="ignore"):
        tmin, tmax = f(f(lo[0] - o[0]) * inv[0]), f(f(hi[0] - o[0]) * inv[0])
        tymin, tymax = f(f(lo[1] - o[1]) * inv[1]), f(f(hi[1] - o[1]) * inv[1])
        if tmin > tymax or tymin > tmax:
            return False
        if tymin > tmin:
            tmin = tymin
        if tymax < tmax:
            tmax = tymax
        tzmin, tzmax = f(f(lo[2] - o[2]) * inv[2]), f(f(hi[2] - o[2]) * inv[2])
        if tmin > tzmax or tzmin > tmax:
            return False
        if tzmax < tmax:
            tmax = tzmax
        return bool(tmax > 0)


def _reference_walk(nodes, o3, inv, neg):
    """box tests and reached leaves, in order, of the reference's stack traversal (basic.cu:156-196)"""
    boxes, leaves, stack, cur = [], [], [], 0
    while True:
        nd = nodes[cur]
        lo = [nd["max"][k] if neg[k] else nd["min"][k] for k in range(3)]
        hi = [nd["min"][k] if neg[k] else nd["max"][k] for k in range(3)]
        hit = _slab(lo, hi, o3, inv)
        boxes.append((tuple(map(float, nd["min"])), tuple(map(float, nd["max"])), hit))
        if hit and nd["count"] > 0:
            leaves.append(int(nd["offset"]))
        if hit and nd["count"] == 0:
            if neg[nd["axis"]]:
                stack.append(cur + 1)
                cur = int(nd["offset"])
            else:
                stack.append(int(nd["offset"]))
                cur = cur + 1
        else:
            if not stack:
                break
            cur = stack.pop()
    return boxes, leaves


def _threaded_walk(T, n, o3, inv, neg):
    """the same, walking the stackless layout: i = hit && inner ? i + 1 : skip"""
    o = sum(1 << k for k in range(3) if neg[k])
    flat = T.reshape(-1)
    boxes, leaves, i = [], [], o * n
    while i != -2147483648:
        r = flat[i]
        lo, hi = list(r["lo"]), [r["hix"], r["hiy"], r["hiz"]]
        hit = _slab(lo, hi, o3, inv)
        mn = tuple(float(hi[k] if neg[k] else lo[k]) for k in range(3))
        mx = tuple(float(lo[k] if neg[k] else hi[k]) for k in range(3))
        boxes.append((mn, mx, hit))
        if hit and r["link"] < 0:
            leaves.append(int(~r["link"]))
        i = i + 1 if (hit and r["link"] >= 0) else int(r["skip"])
        assert i == -2147483648 or o * n <= i < (o + 1) * n
    return boxes, leaves


def _random_ray(rng, trial):
    f = np.float32
    o3 = f(rng.uniform(-6, 6, 3)) + f([0, 2.5, 0])
    d3 = f(rng.normal(size=3))
    if trial % 5 == 0:
        d3[rng.integers(3)] = f(0.0) if trial % 10 == 0 else f(-0.0)
    with np.errstate(all="ignore"):
        inv = f(1.0) / d3
    return o3, inv, [bool(inv[k] < 0) for k in range(3)]


def test_threaded_tree_on_random_trees():
    """Random binary trees in the reference's depth-first layout (random shapes, split axes and -- deliberately --
    boxes that are not nested, so that every hit/miss combination occurs): the stackless walk equals the stack walk."""
    from lens_trace_b200 import capi
    rng = np.random.default_rng(2024)
    for tree in range(12):
        n_leaves = int(rng.integers(1, 40))
        nodes = np.zeros(2 * n_leaves - 1, L.NODE)
        counter = {"i": 0, "prim": 0}

        def build(leaves):
            i = counter["i"]
            counter["i"] += 1
            c = rng.uniform(-4, 4, 3) + [0, 2.5, 0]
            h = rng.uniform(0.2, 4.0, 3)
            nodes["min"][i] = c - h
            nodes["max"][i] = c + h
            if leaves == 1:
                nodes["offset"][i] = counter["prim"]
                nodes["count"][i] = 1 if rng.random() < 0.9 else 2
                counter["prim"] += 1
            else:
                left = int(rng.integers(1, leaves))
                nodes["axis"][i] = int(rng.integers(3))
                build(left)
                nodes["offset"][i] = counter["i"]
                build(leaves - left)

        build(n_leaves)
        n = len(nodes)
        T = capi.build_threaded(nodes)
        for trial in range(30):
            o3, inv, neg = _random_ray(rng, trial)
            assert _threaded_walk(T, n, o3, inv, neg) == _reference_walk(nodes, o3, inv, neg)


def test_threaded_tree_is_the_reference_traversal_order(tmp_path):
    """lt_scene_upload's stackless layout (8 octant copies in visit order, host-built, no GPU needed): walking it
    with `i = hit && inner ? i + 1 : skip` tests the same boxes in the same order and reaches the same leaves in
    the same order as the reference's stack traversal (basic.cu:156-196), for rays of every sign octant
    including axis-parallel ones (+0 / -0 direction components)."""
    from lens_trace_b200 import capi
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 10, 0x5EED)
    scenes = [host.load_scene_buffers(p), util.scene("cornell_box"), util.scene("cornell_box_lens"),
              util.single_triangle_scene(), util.multi_prim_leaf_scene()]
    rng = np.random.default_rng(7)
    f = np.float32
    for sb in scenes:
        nodes = sb.nodes
        n = len(nodes)
        T = capi.build_threaded(nodes)
        assert T.shape == (8, n)
        for o in range(8):  # every copy is a permutation of the nodes, bounds swapped per the octant's signs
            want = sorted((tuple(nd["min"]), tuple(nd["max"])) for nd in nodes)
            got = []
            for r in T[o]:
                lo, hi = list(r["lo"]), [r["hix"], r["hiy"], r["hiz"]]
                mn = [hi[k] if (o >> k) & 1 else lo[k] for k in range(3)]
                mx = [lo[k] if (o >> k) & 1 else hi[k] for k in range(3)]
                got.append((tuple(f(v) for v in mn), tuple(f(v) for v in mx)))
            assert sorted(got) == want
        for trial in range(40):
            o3, inv, neg = _random_ray(rng, trial)
            assert _threaded_walk(T, n, o3, inv, neg) == _reference_walk(nodes, o3, inv, neg)


def test_unreachable_node_entries_are_rejected_on_the_host():
    """validate_tree (lt_scene_upload, lt_debug_build_threaded): every array entry must be reachable from the root."""
    sb = util.scene("cornell_box")
    capi.build_threaded(sb.nodes)
    padded = np.concatenate([sb.nodes, sb.nodes[-1:]])
    with pytest.raises(capi.LtError) as e:
        capi.build_threaded(padded)
    assert "reachable" in str(e.value)


@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "green_wall"])
def test_sah_builder_option(name):
    """ACCELERATION_STRUCTURE_TYPE_SAH_B200: a valid tree in the reference layout over the same primitives, fewer box
    tests per ray than the median split, the same picture except where a ray grazes an edge shared by two triangles."""
    path = os.path.join(util.MODELS, name + ".obj")
    sah = host.load_scene_buffers(path, host.AccelerationStructure.HOST_SAH)
    med = util.scene(name)
    _check_tree(sah)
    assert len(sah.nodes) == len(med.nodes)
    assert sorted(p.tobytes() for p in sah.prims) == sorted(p.tobytes() for p in med.prims)
    assert sah.lights["count"][0] == med.lights["count"][0]
    cam = util.default_camera(0.02)
    a, sa = O.render(L.KERNEL_BASIC_CL, sah, cam, 200, 150, with_stats=True, threads=0)
    b, sb = O.render(L.KERNEL_BASIC_CL, med, cam, 200, 150, with_stats=True, threads=0)
    assert sa.nodeTests <= sb.nodeTests
    assert (np.abs(a - b).max(axis=-1) > 0).mean() < 0.002
    capi.build_threaded(sah.nodes)  # passes the upload-time validation

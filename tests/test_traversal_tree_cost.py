"""The traversal tree is built for the cost of the walk that runs on it: of a SAH sweep tree and a PLOC tree over the
reference's leaves, and the better of the two after treelet restructuring, lt_scene_upload keeps the one whose pruned
copies have the least expected box tests per root-hitting ray, sum over kept records r != root of
SA(nearest kept ancestor of r) / SA(root).  Checked here: the tree is over the reference's leaf records byte for
byte, with exact min/max inner boxes, a valid layout and the same bytes on every build; the cost, restated in NumPy,
is the least of the candidates and never above the SAH sweep tree's; the walk reaches the reference's leaves; and on
a stand-in ray stream the Cornell box needs fewer box tests per ray than a PLOC tree over the primitives (6.90)."""
import os

import numpy as np

import lt_oracle as O
import util
from lens_trace_b200 import capi, host
from test_threaded_prune import _nested_tree, _rays, _walk

f32 = np.float32


def _area(lo, hi):
    d = hi.astype(np.float64) - lo.astype(np.float64)
    return d[..., 0] * d[..., 1] + d[..., 1] * d[..., 2] + d[..., 2] * d[..., 0]


def pruned_cost(nodes):
    """(cost, kept records) of a tree's pruned copies, restated from pruned_keep: an inner node other than the root
    whose children lie inside its box goes when SA(node) > SA(nearest kept ancestor) / 2"""
    n = len(nodes)
    mn, mx, off, cnt = nodes["min"], nodes["max"], nodes["offset"], nodes["count"]
    area = _area(mn, mx)
    keep = np.ones(n, bool)
    anc = np.zeros(n, np.int64)

    def inside(c, m):
        return bool(((mn[m] <= mn[c]) & (mn[c] <= mx[c]) & (mx[c] <= mx[m])).all())

    for i in range(n):
        if cnt[i] > 0:
            continue
        if i > 0:
            keep[i] = not (inside(i + 1, i) and inside(off[i], i) and area[i] > 0.5 * area[anc[i]])
        anc[i + 1] = anc[off[i]] = i if keep[i] else anc[i]
    total = area[anc[1:][keep[1:]]].sum()
    return (total / area[0] if area[0] > 0 else total), int(keep.sum())


def stand_in_rays(sb, w=480, h=270):
    """camera rays of the default camera at w x h and, from every camera hit, one bounce ray in a uniformly sampled
    direction of the hemisphere around the shading normal (seeded): a stand-in for the GI kernel's ray stream.
    Returns (origins, direction reciprocals, whether the ray may walk the pruned copies)."""
    cam = util.default_camera(0.0, 0)
    py, px = np.mgrid[0:h, 0:w]
    fx = (px.astype(f32) / f32(w) - f32(0.5)).astype(f32).reshape(-1)
    fy = (py.astype(f32) / f32(h) - f32(0.5)).astype(f32).reshape(-1)
    pos = cam["pos"][0]
    O3 = np.stack([fx + pos[0], fy + pos[1], np.full_like(fx, pos[2])], axis=1).astype(f32)
    D = np.stack([-fx, -fy, np.full_like(fx, 5.0)], axis=1).astype(f32)
    ids, hit, tuv, _ = O.primary_hits(2, sb, cam, w, h)
    m = hit.reshape(-1) == 1
    t, u, v = (tuv.reshape(-1, 3)[m, k].astype(np.float64)[:, None] for k in range(3))
    p = sb.prims[ids.reshape(-1)[m]]
    nrm = (1 - u - v) * p["na"] + u * p["nb"] + v * p["nc"]
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    rng = np.random.default_rng(1)
    d = rng.normal(size=nrm.shape)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d *= np.sign((d * nrm).sum(axis=1, keepdims=True))
    hp = O3[m] + t * D[m]
    O3 = np.concatenate([O3, (hp + 1e-4 * nrm).astype(f32)])
    D = np.concatenate([D, d.astype(f32)])
    with np.errstate(all="ignore"):
        INV = f32(1.0) / D
    ok = np.isfinite(INV).all(axis=1) & (INV != 0).all(axis=1) & np.isfinite(O3).all(axis=1)
    return O3, INV, ok


def box_tests_per_ray(pruned, full_tests, O3, INV, ok):
    """box tests per ray, root excluded: rays that may walk the pruned copies walk `pruned`, the others keep their
    count on the full copies (full_tests)"""
    tests = full_tests.copy()
    _, _, tests[ok] = _walk(pruned, O3[ok], INV[ok])
    return tests.mean() - 1


def _check_tree(nodes, prim_count):
    r = capi.traversal_tree(nodes, prim_count)
    T = r["nodes"]
    assert T is not None and len(T) == len(nodes)
    # the reference's leaf records, byte for byte, each once
    leaf = lambda a: sorted(a[a["count"] > 0].tobytes()[k:k + 32] for k in range(0, 32 * int((a["count"] > 0).sum()), 32))
    assert leaf(T) == leaf(nodes)
    # inner boxes: the exact min/max of their children
    inner = np.nonzero(T["count"] == 0)[0]
    a, b = inner + 1, T["offset"][inner]
    np.testing.assert_array_equal(T["min"][inner], np.minimum(T["min"][a], T["min"][b]))
    np.testing.assert_array_equal(T["max"][inner], np.maximum(T["max"][a], T["max"][b]))
    capi.build_threaded(T)  # validate_tree: raises on a malformed layout
    # deterministic, and what the upload walks
    again = capi.traversal_tree(nodes, prim_count)
    assert again["nodes"].tobytes() == T.tobytes()
    assert all(again[k] == r[k] for k in ("reference", "sah", "ploc", "restructured"))
    up = capi.build_traversal_tree(nodes, prim_count)
    assert up["traversal"]
    assert up["pruned"].tobytes() == capi.build_traversal_tree(nodes, prim_count)["pruned"].tobytes()
    assert up["pruned"].tobytes() == capi.build_threaded_pruned(T).tobytes()
    # the cost: restated, the least of the candidates, never above the SAH sweep tree's
    cost, kept = pruned_cost(T)
    assert kept == up["stride"]
    cands = [r["sah"], r["ploc"], r["restructured"]]
    assert abs(cost - min(cands)) <= 1e-9 * cost
    assert cost <= r["sah"] * (1 + 1e-12)
    ref_cost, _ = pruned_cost(nodes)
    assert abs(ref_cost - r["reference"]) <= 1e-9 * ref_cost
    return r, up


def _scenes(tmp_path):
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 10, 0x5EED)
    return [util.scene("cornell_box"), util.scene("cornell_box_lens"), util.scene("green_wall"),
            host.load_scene_buffers(p)]


def test_shipped_models_get_the_cheapest_tree_over_their_leaves(tmp_path):
    for sb in _scenes(tmp_path):
        _check_tree(sb.nodes, len(sb.prims))


def test_random_nested_trees_get_the_cheapest_tree_over_their_leaves():
    rng = np.random.default_rng(17)
    restructured = 0
    for tree in range(12):
        nodes = _nested_tree(rng, int(rng.integers(2, 400)))
        r, up = _check_tree(nodes, int(nodes["offset"][nodes["count"] > 0].max()) + 1)
        restructured += r["restructured"] < min(r["sah"], r["ploc"])
        # the walk reaches the reference's leaves, ray by ray
        O3, INV = _rays(nodes, rng, 2000)
        for exact in (False, True):
            lf, cf, _ = _walk(up["full"], O3, INV, exact)
            lt, ct, _ = _walk(up["pruned"], O3, INV, exact)
            np.testing.assert_array_equal(ct, cf)
            for a, b in zip(np.split(lf, np.cumsum(cf)[:-1]), np.split(lt, np.cumsum(ct)[:-1])):
                assert sorted(a) == sorted(b)
    assert restructured > 0


def test_stand_in_box_tests_per_ray():
    got = {}
    for name in ("cornell_box", "cornell_box_lens"):
        sb = util.scene(name)
        O3, INV, ok = stand_in_rays(sb)
        _, _, full_tests = _walk(capi.build_threaded(sb.nodes), O3, INV)
        got[name] = box_tests_per_ray(capi.build_traversal_tree(sb.nodes, len(sb.prims))["pruned"], full_tests, O3,
                                      INV, ok)
    print("stand-in box tests per ray: %s" % got)
    assert got["cornell_box"] < 6.90  # a PLOC tree over the primitives
    assert got["cornell_box_lens"] < 11.52  # the SAH sweep tree over the leaves


def test_containment_violation_gets_no_traversal_tree():
    sb = util.scene("cornell_box")
    nodes = sb.nodes.copy()
    leaf = int(np.nonzero(nodes["count"] > 0)[0][3])
    nodes["max"][leaf][0] = f32(nodes["max"][0][0] + f32(1))
    r = capi.traversal_tree(nodes, len(sb.prims))
    assert r["nodes"] is None and r["sah"] is None and r["restructured"] is None
    assert abs(r["reference"] - pruned_cost(nodes)[0]) <= 1e-9 * r["reference"]
    up = capi.build_traversal_tree(nodes, len(sb.prims))
    assert not up["traversal"]
    assert up["pruned"].tobytes() == capi.build_threaded_pruned(nodes).tobytes()

"""Traversal tree: the pruned threaded copies of a small scene are built from a SAH tree over the reference's leaves
when every leaf box lies inside all its ancestors' boxes.  A ray with finite, nonzero direction reciprocals and a
finite origin then reaches exactly the leaves the reference reaches, in another order, and the least (t, rank) --
rank = the leaf's position in the reference's visit order of the ray's octant -- is the reference's closest hit.
Walked in float32 with the kernels' arithmetic (_walk), per ray: the same set of leaves as the reference's full
copies, and the same hit."""
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L
from test_threaded_prune import _nested_tree, _rays, _walk

f32 = np.float32


def _fma(a, b, c):
    # float32 a * b is exact in float64; one rounding of the sum, then to float32 (deterministic, which is all the
    # comparison of two orders needs)
    return (a.astype(np.float64) * b + c).astype(f32)


def _dot3z(ax, ay, az, bx, by, bz):
    return (_fma(az, bz, _fma(ax, bx, (ay * by).astype(f32))) + f32(0)).astype(f32)


def _tri(prims, idx, o, d, eps):
    """tri_test's arithmetic for one ray against primitives idx: (accepted before the t comparison, t, u, v)"""
    p = prims[idx]
    a = p["a"].astype(f32)
    e1 = (p["b"].astype(f32) - a).astype(f32)
    e2 = (p["c"].astype(f32) - a).astype(f32)
    pv = np.stack([_fma(d[1], e2[:, 2], -(d[2] * e2[:, 1]).astype(f32)),
                   _fma(d[2], e2[:, 0], -(d[0] * e2[:, 2]).astype(f32)),
                   _fma(d[0], e2[:, 1], -(d[1] * e2[:, 0]).astype(f32))], axis=1)
    det = _dot3z(e1[:, 0], e1[:, 1], e1[:, 2], pv[:, 0], pv[:, 1], pv[:, 2])
    with np.errstate(all="ignore"):
        inv = (f32(1) / det).astype(f32)
        tv = (o - a).astype(f32)
        u = (_dot3z(tv[:, 0], tv[:, 1], tv[:, 2], pv[:, 0], pv[:, 1], pv[:, 2]) * inv).astype(f32)
        q = np.stack([_fma(tv[:, 1], e1[:, 2], -(tv[:, 2] * e1[:, 1]).astype(f32)),
                      _fma(tv[:, 2], e1[:, 0], -(tv[:, 0] * e1[:, 2]).astype(f32)),
                      _fma(tv[:, 0], e1[:, 1], -(tv[:, 1] * e1[:, 0]).astype(f32))], axis=1)
        v = (_dot3z(np.full(len(idx), d[0], f32), np.full(len(idx), d[1], f32), np.full(len(idx), d[2], f32),
                    q[:, 0], q[:, 1], q[:, 2]) * inv).astype(f32)
        t = (_dot3z(e2[:, 0], e2[:, 1], e2[:, 2], q[:, 0], q[:, 1], q[:, 2]) * inv).astype(f32)
        ok = ~(np.abs(det) < eps) & ~((u < 0) | (u > 1)) & ~((v < 0) | ((u + v).astype(f32) > 1))
    return ok, t, u, v


def _closest(prims, seq, o, d, t_init, rank=None):
    """tri_test applied along the leaf sequence seq: strict t < best, and with `rank` the (t, rank) tie-break"""
    best = (0, t_init, 0.0, 0.0, 0)  # prim, t, u, v, hit
    if len(seq) == 0:
        return best
    ok, t, u, v = _tri(prims, seq, o, d, f32(float.fromhex("0x1.a36e30p-14")))
    for k, p in enumerate(seq):
        if not ok[k]:
            continue
        take = t[k] < best[1]
        if rank is not None and t[k] == best[1] and best[4]:
            take = rank[p] < rank[best[0]]
        if take:
            best = (int(p), t[k], u[k], v[k], 1)
    return best


def _per_ray(leaves, counts):
    return np.split(leaves, np.cumsum(counts)[:-1])


def _stand_in_rays(sb, w=96, h=54):
    """camera rays of the default camera, a bounce ray from each camera hit (origin on the surface, ignoring the hit
    primitive), and rays aimed at the vertices and edge midpoints of every triangle"""
    cam = util.default_camera(0.0, 0)
    py, px = np.mgrid[0:h, 0:w]
    fx = (px.astype(f32) / f32(w) - f32(0.5)).astype(f32).reshape(-1)
    fy = (py.astype(f32) / f32(h) - f32(0.5)).astype(f32).reshape(-1)
    pos = cam["pos"][0]
    O3 = np.stack([fx + pos[0], fy + pos[1], np.full_like(fx, pos[2])], axis=1).astype(f32)
    D = np.stack([-fx, -fy, np.full_like(fx, 5.0)], axis=1).astype(f32)
    ign = np.full(len(O3), -1)
    ids, hit, tuv, _ = O.primary_hits(2, sb, cam, w, h)
    m = hit.reshape(-1) == 1
    t = tuv.reshape(-1, 3)[m, 0].astype(f32)[:, None]
    hp = (O3[m] + t * D[m]).astype(f32)
    rng = np.random.default_rng(4)
    d = rng.normal(size=hp.shape).astype(f32)
    P = sb.prims
    targets = np.concatenate([P["a"], P["b"], P["c"], (P["a"] + P["b"]) / 2, (P["b"] + P["c"]) / 2,
                              (P["c"] + P["a"]) / 2]).astype(f32)
    src = np.asarray(pos, f32) + rng.normal(scale=3.0, size=targets.shape).astype(f32)
    O3 = np.concatenate([O3, hp, src])
    D = np.concatenate([D, d, (targets - src).astype(f32)])
    ign = np.concatenate([ign, ids.reshape(-1)[m], np.full(len(src), -1)])
    return O3, D, ign


def _check_scene(sb, rng, n_random=3000):
    prims = sb.prims
    r = capi.build_traversal_tree(sb.nodes, len(prims))
    assert r["traversal"]
    assert r["pruned"].shape[1] <= len(sb.nodes)
    np.testing.assert_array_equal(r["full"], capi.build_threaded(sb.nodes))
    O3, D, ign = _stand_in_rays(sb)
    Or, INVr = _rays(sb.nodes, rng, n_random)
    with np.errstate(all="ignore"):
        INV = (f32(1) / D).astype(f32)
    O3 = np.concatenate([O3, Or])
    INV = np.concatenate([INV, INVr])
    with np.errstate(all="ignore"):
        D = np.concatenate([D, (f32(1) / INVr).astype(f32)])
    ign = np.concatenate([ign, np.full(len(Or), -1)])
    ok = np.isfinite(INV).all(axis=1) & (INV != 0).all(axis=1) & np.isfinite(O3).all(axis=1)
    O3, INV, D, ign = O3[ok], INV[ok], D[ok], ign[ok]
    oct_ = (INV[:, 0] < 0) * 1 + (INV[:, 1] < 0) * 2 + (INV[:, 2] < 0) * 4
    ties = 0
    for exact in (False, True):
        lf, cf, _ = _walk(r["full"], O3, INV, exact)
        lt, ct, _ = _walk(r["pruned"], O3, INV, exact)
        np.testing.assert_array_equal(ct, cf)
        for i, (a, b) in enumerate(zip(_per_ray(lf, cf), _per_ray(lt, ct))):
            assert sorted(a) == sorted(b), i
            if exact:
                continue
            a, b = a[a != ign[i]], b[b != ign[i]]
            want = _closest(prims, a, O3[i], D[i], f32(3.4028235e38))
            got = _closest(prims, b, O3[i], D[i], f32(3.4028235e38), r["rank"][oct_[i]])
            assert util.bits(np.array(got[1:4], f32)).tolist() == util.bits(np.array(want[1:4], f32)).tolist(), i
            assert (got[0], got[4]) == (want[0], want[4]), i
            # ranks follow the reference's order: the reference's own sequence is sorted by them
            np.testing.assert_array_equal(np.diff(r["rank"][oct_[i]][a]) > 0, True)
            ties += _closest(prims, b, O3[i], D[i], f32(3.4028235e38))[0] != want[0]
    return r, ties


def test_traversal_tree_reaches_the_reference_leaves_and_hits(tmp_path):
    rng = np.random.default_rng(21)
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 10, 0x5EED)
    for sb in (util.scene("cornell_box"), util.scene("cornell_box_lens"), util.scene("green_wall"),
               host.load_scene_buffers(p)):
        _check_scene(sb, rng)


def test_random_nested_trees_get_a_traversal_tree():
    rng = np.random.default_rng(6)
    for tree in range(10):
        nodes = _nested_tree(rng, int(rng.integers(2, 80)))
        r = capi.build_traversal_tree(nodes, int(nodes["offset"][nodes["count"] > 0].max()) + 1)
        assert r["traversal"]
        O3, INV = _rays(nodes, rng, 3000)
        for exact in (False, True):
            lf, cf, _ = _walk(r["full"], O3, INV, exact)
            lt, ct, _ = _walk(r["pruned"], O3, INV, exact)
            np.testing.assert_array_equal(ct, cf)
            for a, b in zip(_per_ray(lf, cf), _per_ray(lt, ct)):
                assert sorted(a) == sorted(b)


def _quad_grid():
    """a wall of quads split along their diagonals, and pairs of coincident triangles in front of it (the second of
    each pair emissive, so the two materials differ), in view of the default camera"""
    tris = []
    for i in range(6):
        for j in range(6):
            x0, y0 = -4.5 + 1.5 * i, -2.0 + 1.5 * j
            a, b, c, d = (x0, y0, 3.0), (x0 + 1.5, y0, 3.0), (x0 + 1.5, y0 + 1.5, 3.0), (x0, y0 + 1.5, 3.0)
            tris += [(a, b, c), (a, c, d)]
    pairs = []
    for k in range(10):
        x0, y0, z0 = -4.0 + 0.8 * k, -1.5 + 0.6 * (k % 5), -1.0 - 0.3 * k
        t = ((x0, y0, z0), (x0 + 1.0, y0 + 0.2, z0 + 0.1 * (k % 3)), (x0 + 0.3, y0 + 1.1, z0 - 0.1 * (k % 2)))
        pairs.append(t)
    return tris, pairs


def _tie_scene(path):
    tris, pairs = _quad_grid()
    base = os.path.splitext(path)[0]
    with open(base + ".mtl", "w") as f:
        f.write("newmtl M\nKd 0.5 0.5 0.5\nnewmtl N\nKd 0.2 0.7 0.3\nnewmtl E\nKd 1 1 1\nKe 4 4 4\n")
    with open(path, "w") as f:
        f.write("mtllib %s.mtl\n" % os.path.basename(base))
        k = 0
        for mtl, t in [("M", t) for t in tris] + [(m, t) for t in pairs for m in ("M", "N")] + \
                [("E", ((-2.0, 6.0, -2.0), (2.0, 6.0, -2.0), (0.0, 6.0, 2.0)))]:
            f.write("usemtl %s\n" % mtl)
            for v in t:
                f.write("v %r %r %r\n" % tuple(float(x) for x in v))
            f.write("f %d %d %d\n" % (3 * k + 1, 3 * k + 2, 3 * k + 3))
            k += 1
    return host.load_scene_buffers(path)


def _tied_pairs(sb):
    """(leaf of the first, leaf of the second) primitive of each coincident pair, as primitive indices"""
    key = {}
    for i, p in enumerate(sb.prims):
        key.setdefault(p["a"].tobytes() + p["b"].tobytes() + p["c"].tobytes(), []).append(i)
    return [v for v in key.values() if len(v) == 2]


def test_tie_scene_keeps_the_reference_primitive(tmp_path):
    sb = _tie_scene(str(tmp_path / "ties.obj"))
    pairs = _tied_pairs(sb)
    assert len(pairs) == 10
    r = capi.build_traversal_tree(sb.nodes, len(sb.prims))
    assert r["traversal"]
    # the test has teeth: some octant visits the two leaves of a tied pair in the other order on the traversal tree
    swapped = 0
    for o in range(8):
        seq_ref = [~v for v in r["full"][o]["link"] if v < 0]
        seq_trav = [~v for v in r["pruned"][o]["link"] if v < 0]
        for a, b in pairs:
            swapped += (seq_ref.index(a) < seq_ref.index(b)) != (seq_trav.index(a) < seq_trav.index(b))
    assert swapped > 0
    _, ties = _check_scene(sb, np.random.default_rng(9), 1000)
    assert ties > 0  # without the tie-break some ray would end on the other primitive


def test_containment_violation_takes_the_reference_pruned_copies():
    rng = np.random.default_rng(12)
    sb = util.scene("cornell_box")
    for case in range(4):
        nodes = sb.nodes.copy()
        leaf = int(rng.choice(np.nonzero(nodes["count"] > 0)[0]))
        if case == 0:  # a leaf pokes out of its ancestors
            nodes["max"][leaf][0] = f32(nodes["max"][0][0] + f32(1))
        elif case == 1:  # NaN bound
            nodes["min"][leaf][1] = f32(np.nan)
        elif case == 2:  # two leaves link one primitive
            other = int(np.nonzero(nodes["count"] > 0)[0][0 if leaf != np.nonzero(nodes["count"] > 0)[0][0] else 1])
            nodes["offset"][leaf] = nodes["offset"][other]
        else:  # inverted bounds
            nodes["min"][leaf][2], nodes["max"][leaf][2] = nodes["max"][leaf][2], nodes["min"][leaf][2] - f32(1)
        r = capi.build_traversal_tree(nodes, len(sb.prims))
        assert not r["traversal"] and r["rank"] is None, case
        want = capi.build_threaded_pruned(nodes)
        assert r["pruned"].tobytes() == want.tobytes(), case
        assert r["full"].tobytes() == capi.build_threaded(nodes).tobytes(), case
    leaf_root = util.single_triangle_scene()
    assert not capi.build_traversal_tree(leaf_root.nodes, 1)["traversal"]


# ---- GPU ----

@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.mark.gpu
def test_tie_scene_equals_the_oracle_on_every_schedule(ctx, tmp_path):
    from test_gpu_parity import FLAVOUR, assert_images_match
    sb = _tie_scene(str(tmp_path / "ties.obj"))
    sc = ctx.upload(sb)
    assert ctx.uses_traversal_tree(sc)
    for yaw in (0.0, 0.03):
        cam = util.default_camera(yaw, 1)
        for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_GI):
            ids, hit, tuv = ctx.primary_hits(sc, cam, kernel, 320, 180)
            oids, ohit, otuv, _ = O.primary_hits(FLAVOUR[kernel], sb, cam, 320, 180)
            np.testing.assert_array_equal(hit, ohit)
            np.testing.assert_array_equal(ids, oids)
            util.assert_bit_equal(tuv, otuv, "tie scene t,u,v")
        want = O.render(L.KERNEL_BASIC_CU, sb, cam, 320, 180, threads=0)
        util.assert_bit_equal(ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, 320, 180)), want, "basic")
        for kernel in (L.KERNEL_ACCUMULATOR, L.KERNEL_GI):
            want = O.render(kernel, sb, cam, 160, 96, max_ray_depth=4, threads=0)
            for flags in (L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT):
                got = ctx.render(sc, cam, capi.make_params(kernel, 160, 96, max_ray_depth=4, flags=flags))
                assert_images_match(got, want, "tie scene kernel %d flags %d" % (kernel, flags), max_outliers=3)
    sc.release()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "green_wall"])
def test_shipped_models_use_the_traversal_tree(ctx, name):
    sc = ctx.upload(util.scene(name))
    assert ctx.uses_traversal_tree(sc)
    sc.release()
    ctx.debug_limits(0, 100000)  # device-built copies: no traversal tree
    sc = ctx.upload(util.scene(name))
    assert not ctx.uses_traversal_tree(sc)
    sc.release()
    ctx.debug_limits(65536, 100000)

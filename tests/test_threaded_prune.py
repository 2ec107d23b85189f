"""Pruned threaded copies: the eight octant sequences without the inner nodes whose child boxes lie inside their own
box.  Walked in float32 with the kernels' arithmetic (FSUB, FMUL, then max/min or the select chain), they must
record the same leaves in the same order as the full copies for every ray with finite, nonzero direction
reciprocals and a finite origin -- the rays trav_begin_threaded sends to them."""
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L

DONE = -2147483648
f32 = np.float32


def _walk(T, O3, INV, exact=False):
    """Walks copies T (8 x stride records, skip links index T flattened) for rays (O3, INV), all lanes at once.
    Returns (leaves in ray-major order, leaves per ray, box tests per ray)."""
    stride = T.shape[1]
    flat = T.reshape(-1)
    lo = np.ascontiguousarray(flat["lo"], dtype=f32)
    hi = np.stack([flat["hix"], flat["hiy"], flat["hiz"]], axis=1).astype(f32)
    link, skip = flat["link"].astype(np.int64), flat["skip"].astype(np.int64)
    oct_ = (INV[:, 0] < 0) * 1 + (INV[:, 1] < 0) * 2 + (INV[:, 2] < 0) * 4
    R = len(O3)
    cur = oct_.astype(np.int64) * stride
    tests = np.zeros(R, np.int64)
    events = []
    active = np.ones(R, bool)
    with np.errstate(all="ignore"):
        while active.any():
            idx = np.nonzero(active)[0]
            c = cur[idx]
            assert ((c >= oct_[idx] * stride) & (c < (oct_[idx] + 1) * stride)).all()
            t0 = (lo[c] - O3[idx]) * INV[idx]  # float32 FSUB then FMUL, no contraction
            t1 = (hi[c] - O3[idx]) * INV[idx]
            if exact:  # select chain of basic.cu:136-154 on the pre-selected bounds
                tx0, ty0, tz0, tx1, ty1, tz1 = t0[:, 0], t0[:, 1], t0[:, 2], t1[:, 0], t1[:, 1], t1[:, 2]
                miss1 = (tx0 > ty1) | (ty0 > tx1)
                a = np.where(ty0 > tx0, ty0, tx0)
                b = np.where(ty1 < tx1, ty1, tx1)
                miss2 = (a > tz1) | (tz0 > b)
                hit = ~miss1 & ~miss2 & (np.where(tz1 < b, tz1, b) > 0)
            else:
                a = np.fmax(np.fmax(t0[:, 0], t0[:, 1]), t0[:, 2])
                b = np.fmin(np.fmin(t1[:, 0], t1[:, 1]), t1[:, 2])
                hit = (a <= b) & (b > 0)
            tests[idx] += 1
            lk = link[c]
            ev = np.full(R, -1, np.int64)
            leaf = hit & (lk < 0)
            ev[idx[leaf]] = ~lk[leaf]
            events.append(ev)
            nxt = np.where(hit & (lk >= 0), c + 1, skip[c])
            cur[idx] = nxt
            active[idx] = nxt != DONE
    E = np.stack(events).T
    return E[E >= 0], (E >= 0).sum(axis=1), tests


def _rays(nodes, rng, n):
    """Finite rays with finite, nonzero reciprocals: origins around the scene, inside node boxes and exactly on box
    planes; directions with one or two tiny components among them."""
    mn, mx = nodes["min"].astype(np.float64), nodes["max"].astype(np.float64)
    finite = np.isfinite(mn).all(axis=1) & np.isfinite(mx).all(axis=1)
    mn, mx = mn[finite], mx[finite]
    lo, hi = mn.min(axis=0), mx.max(axis=0)
    ext = np.maximum(hi - lo, 1.0)
    O3 = rng.uniform(lo - ext, hi + ext, (n, 3))
    k = rng.integers(len(mn), size=n)
    inside = rng.uniform(mn[k], mx[k])
    third = n // 3
    O3[:third] = inside[:third]  # inside a box
    plane = inside[third:2 * third].copy()  # exactly on a box plane
    ax = rng.integers(3, size=len(plane))
    side = rng.random(len(plane)) < 0.5
    kk = k[third:2 * third]
    plane[np.arange(len(plane)), ax] = np.where(side, mn[kk, ax], mx[kk, ax])
    O3[third:2 * third] = plane
    O3 = O3.astype(f32)
    D = rng.normal(size=(n, 3))
    tiny = rng.random(n) < 0.3
    for col_choice in range(2):  # one or two tiny components
        col = rng.integers(3, size=n)
        mag = 10.0 ** rng.uniform(-37, -4, n) * np.where(rng.random(n) < 0.5, -1, 1)
        sel = tiny & ((col_choice == 0) | (rng.random(n) < 0.5))
        D[sel, col[sel]] = mag[sel]
    D = D.astype(f32)
    with np.errstate(all="ignore"):
        INV = f32(1.0) / D
    ok = np.isfinite(INV).all(axis=1) & (INV != 0).all(axis=1) & np.isfinite(O3).all(axis=1)
    return O3[ok], INV[ok]


def _check_same_leaves(nodes, rng, n_rays=6000):
    full = capi.build_threaded(nodes)
    pruned = capi.build_threaded_pruned(nodes)
    O3, INV = _rays(nodes, rng, n_rays)
    assert len(O3) > n_rays // 2
    for exact in (False, True):
        lf, cf, tf = _walk(full, O3, INV, exact)
        lp, cp, tp = _walk(pruned, O3, INV, exact)
        np.testing.assert_array_equal(cp, cf)
        np.testing.assert_array_equal(lp, lf)
    return full, pruned


def _check_records(nodes, pruned):
    """Every pruned copy holds every leaf exactly once; skip links stay in their copy and lead forward."""
    stride = pruned.shape[1]
    leaves = sorted(int(nd["offset"]) for nd in nodes if nd["count"] > 0)
    for o in range(8):
        rec = pruned[o]
        assert sorted(int(~v) for v in rec["link"] if v < 0) == leaves
        skip = rec["skip"].astype(np.int64)
        pos = o * stride + np.arange(stride)
        ok = (skip == DONE) | ((skip > pos) & (skip < (o + 1) * stride))
        assert ok.all(), o
        lo = [nodes["max"][0][k] if (o >> k) & 1 else nodes["min"][0][k] for k in range(3)]
        np.testing.assert_array_equal(rec["lo"][0], np.array(lo, f32))  # the root stays first


def _nested_tree(rng, n_leaves):
    """A random tree in the reference's depth-first layout whose inner boxes are the exact min/max of their children."""
    nodes = np.zeros(2 * n_leaves - 1, L.NODE)
    counter = {"i": 0, "prim": 0}

    def build(leaves):
        i = counter["i"]
        counter["i"] += 1
        if leaves == 1:
            c = rng.uniform(-8, 8, 3)
            h = rng.uniform(0.05, 3.0, 3)
            nodes["min"][i], nodes["max"][i] = f32(c - h), f32(c + h)
            nodes["offset"][i] = counter["prim"]
            nodes["count"][i] = 1
            counter["prim"] += 1
            return
        left = int(rng.integers(1, leaves))
        nodes["axis"][i] = int(rng.integers(3))
        build(left)
        nodes["offset"][i] = counter["i"]
        build(leaves - left)
        a, b = i + 1, int(nodes["offset"][i])
        nodes["min"][i] = np.minimum(nodes["min"][a], nodes["min"][b])
        nodes["max"][i] = np.maximum(nodes["max"][a], nodes["max"][b])

    build(n_leaves)
    return nodes


def _kept(pruned, box_min, box_max):
    """is a record with these bounds (compared bitwise: NaN included) in octant copy 0 (lo = min, hi = max)?"""
    rec = pruned[0]
    lo = np.ascontiguousarray(rec["lo"], f32).view(np.uint32)
    hi = np.stack([rec["hix"], rec["hiy"], rec["hiz"]], axis=1).astype(f32).view(np.uint32)
    mn, mx = np.asarray(box_min, f32).view(np.uint32), np.asarray(box_max, f32).view(np.uint32)
    return bool(((lo == mn).all(axis=1) & (hi == mx).all(axis=1)).any())


def test_pruned_copies_record_the_same_leaves_on_the_shipped_models(tmp_path):
    rng = np.random.default_rng(11)
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 10, 0x5EED)
    scenes = [util.scene("cornell_box"), util.scene("cornell_box_lens"), util.scene("green_wall"),
              host.load_scene_buffers(p), util.single_triangle_scene(), util.multi_prim_leaf_scene()]
    for name in ("cornell_box", "cornell_box_lens", "green_wall"):
        scenes.append(host.load_scene_buffers(os.path.join(util.MODELS, name + ".obj"), host.AccelerationStructure.HOST_SAH))
    for sb in scenes:
        full, pruned = _check_same_leaves(sb.nodes, rng)
        _check_records(sb.nodes, pruned)
        assert pruned.shape[1] <= full.shape[1]
    assert capi.build_threaded_pruned(util.scene("cornell_box").nodes).shape == (8, 55)  # of 83 records


def test_pruned_copies_on_random_nested_trees():
    rng = np.random.default_rng(5)
    dropped = 0
    for tree in range(10):
        nodes = _nested_tree(rng, int(rng.integers(2, 60)))
        full, pruned = _check_same_leaves(nodes, rng, 3000)
        _check_records(nodes, pruned)
        dropped += full.shape[1] - pruned.shape[1]
    assert dropped > 0


def test_containment_violation_keeps_the_node():
    """A child that pokes out of its parent's box: the parent is kept, and the leaves stay the same."""
    rng = np.random.default_rng(8)
    checked = 0
    for tree in range(20):
        nodes = _nested_tree(rng, 40)
        pruned = capi.build_threaded_pruned(nodes)
        inner = [i for i in range(1, len(nodes)) if nodes["count"][i] == 0]
        gone = [i for i in inner if not _kept(pruned, nodes["min"][i], nodes["max"][i])]
        if not gone:
            continue
        m = gone[0]
        c = m + 1 if rng.random() < 0.5 else int(nodes["offset"][m])
        ax = int(rng.integers(3))
        nodes["max"][c][ax] = f32(nodes["max"][m][ax] + f32(0.5))
        full, pruned = _check_same_leaves(nodes, rng, 3000)
        _check_records(nodes, pruned)
        assert _kept(pruned, nodes["min"][m], nodes["max"][m])
        nodes["min"][m][ax] = f32(np.nan)  # NaN bounds never count as containing
        assert _kept(capi.build_threaded_pruned(nodes), nodes["min"][m], nodes["max"][m])
        checked += 1
    assert checked >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "green_wall"])
def test_gi_on_full_copies_equals_pruned(name):
    """GI launches on the full threaded copies only (test hook) equal the default launches bit for bit, on every
    schedule; the LBVH tree of the same model passes the CPU walk check."""
    ctx = capi.Context(0)
    sb = util.scene(name)
    sc = ctx.upload(sb)
    cam = util.default_camera(0.02, 1)
    for flags in (0, L.FLAG_WAVEFRONT, L.FLAG_MEGAKERNEL):
        params = capi.make_params(L.KERNEL_GI, 480, 270, max_ray_depth=4, frames=2, flags=flags)
        ctx.debug_full_threaded(sc, False)
        got = ctx.render(sc, cam, params)
        ctx.debug_full_threaded(sc, True)
        full = ctx.render(sc, cam, params)
        util.assert_bit_equal(got, full, "%s flags %d" % (name, flags))
    ctx.debug_full_threaded(sc, False)
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 320, 180)
    oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, 320, 180)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv, "%s primary t,u,v" % name)
    sc.release()
    lb = ctx.build_lbvh(sb.prims, sb.materials)
    lbvh, _ = ctx.download(lb)
    lb.release()
    _check_same_leaves(lbvh.nodes, np.random.default_rng(3))
    ctx.close()

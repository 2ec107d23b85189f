"""lt_scene_refit / lt_scene_refit_device on the GPU: the refitted nodes equal the NumPy restatement
(tests/test_scene_refit.py) byte for byte, and every render entry point on a refitted scene equals, bit for bit, the
same call on a scene uploaded fresh from the refitted nodes, the new primitives and the scene's materials and lights.

Deformations are deterministic: one object of the Cornell and lens scenes translated or scaled, a sine displacement of
the synthetic mesh."""
import ctypes as C
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L
from test_scene_refit import restate_refit, positive_zeros

pytestmark = pytest.mark.gpu

KERNELS = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY, L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR,
           L.KERNEL_GI25, L.KERNEL_GI]
FLAGS = [0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_NO_THREADED, L.FLAG_NO_STREAM, L.FLAG_WAVEFRONT | L.FLAG_SERIAL]
GI_PLUGIN = os.path.join(util.ROOT, "tests", "plugins", "gi_plugin.cu")


def interior(prims):
    """the primitives of the objects inside the Cornell room (not its walls, floor or ceiling)"""
    lo = np.minimum(np.minimum(prims["a"], prims["b"]), prims["c"])
    hi = np.maximum(np.maximum(prims["a"], prims["b"]), prims["c"])
    sel = (lo[:, 0] > -2.4) & (hi[:, 0] < 2.4) & (lo[:, 2] > -2.4) & (hi[:, 2] < 2.4) & (hi[:, 1] > 0.01) & \
        (hi[:, 1] < 4.9)
    assert sel.any() and not sel.all()
    return sel


def translated(prims, by=(0.3, 0.2, -0.25)):
    out = prims.copy()
    sel = interior(prims)
    for k in ("a", "b", "c"):
        out[k][sel] += np.asarray(by, np.float32)
    return out


def scaled(prims, s=1.1):
    out = prims.copy()
    sel = interior(prims)
    centre = np.concatenate([prims[k][sel] for k in ("a", "b", "c")]).mean(axis=0).astype(np.float32)
    for k in ("a", "b", "c"):
        out[k][sel] = (out[k][sel] - centre) * np.float32(s) + centre
    return out


def sine(prims, amp=0.02, phase=0.0):
    out = prims.copy()
    for k in ("a", "b", "c"):
        v = out[k].astype(np.float64)
        v[:, 1] += amp * np.sin(3.0 * v[:, 0] + 2.0 * v[:, 2] + phase)
        out[k] = v.astype(np.float32)
    return out


DEFORM = {"cornell_box": translated, "cornell_box_lens": scaled}


def fresh(ctx, scene, sb):
    """a scene uploaded from the refitted scene's buffers"""
    down, _ = ctx.download(scene)
    return ctx.upload(L.SceneBuffers(down.nodes, down.prims, sb.materials, down.lights))


def download(ctx, scene):
    down, _ = ctx.download(scene)
    return down


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def synth1m(ctx, tmp_path_factory):
    """the synthetic 1 M-triangle mesh (grid 707: 999 710 triangles, 1 999 419 nodes), uploaded"""
    p = str(tmp_path_factory.mktemp("synth") / "synth707.obj")
    host.write_synthetic_scene(p, 707, 0x5EED)
    sb = host.load_scene_buffers(p)
    sc = ctx.upload(sb)
    yield sb, sc
    sc.release()


def check_nodes(ctx, sc, nodes, prims, what):
    ctx.refit(sc, prims)
    down = download(ctx, sc)
    assert down.prims.tobytes() == prims.tobytes(), what
    want = restate_refit(nodes, prims)
    assert down.nodes.tobytes() == want.tobytes(), what
    return down


@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "multi_prim_leaf"])
def test_refit_nodes_equal_restatement(ctx, name):
    sb = util.multi_prim_leaf_scene() if name == "multi_prim_leaf" else util.scene(name)
    sc = ctx.upload(sb)
    prims = sine(sb.prims, 0.1) if name == "multi_prim_leaf" else DEFORM[name](sb.prims)
    check_nodes(ctx, sc, sb.nodes, prims, name)
    assert ctx.stats().upload_ms > 0.0
    # the refit is deterministic: the same input twice gives the same bytes
    first = download(ctx, sc).nodes.tobytes()
    ctx.refit(sc, prims)
    assert download(ctx, sc).nodes.tobytes() == first
    sc.release()


def test_refit_nodes_of_a_ploc_scene(ctx):
    sb = util.scene("cornell_box_lens")
    sc = ctx.build_ploc(sb.prims, sb.materials)
    built = download(ctx, sc)  # the built scene's primitive order
    check_nodes(ctx, sc, built.nodes, scaled(built.prims), "PLOC scene")
    sc.release()


def test_refit_nodes_of_the_1m_mesh(ctx, synth1m):
    sb, sc = synth1m
    check_nodes(ctx, sc, sb.nodes, sine(sb.prims), "1 M mesh")
    ctx.refit(sc, sb.prims)


def check_renders(ctx, a, b, kernels, flags, size=(96, 64), what=""):
    w, h = size
    for kernel in kernels:
        for f in flags:
            cam = util.default_camera(0.03, 2)
            for frames, mode in ((1, L.ACCUM_NONE), (3, L.ACCUM_RUNNING_MEAN)):
                p = capi.make_params(kernel, w, h, max_ray_depth=3, frames=frames, accum_mode=mode, flags=f)
                ctx.accum_reset()
                got = ctx.render(a, cam, p)
                ctx.accum_reset()
                want = ctx.render(b, cam, p)
                util.assert_bit_equal(got, want, "%s kernel %d flags %d frames %d" % (what, kernel, f, frames))
    cam = util.default_camera(0.03)
    for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_GI):
        for got, want in zip(ctx.primary_hits(a, cam, kernel, w, h), ctx.primary_hits(b, cam, kernel, w, h)):
            assert got.tobytes() == want.tobytes(), "%s primary hits, kernel %d" % (what, kernel)


@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens"])
def test_refit_renders_equal_fresh_upload(ctx, name):
    sb = util.scene(name)
    sc = ctx.upload(sb)
    ctx.refit(sc, DEFORM[name](sb.prims))
    ref = fresh(ctx, sc, sb)
    assert ctx.uses_traversal_tree(sc) == ctx.uses_traversal_tree(ref)
    check_renders(ctx, sc, ref, KERNELS, FLAGS, what=name)
    # lt_render_device into a torch tensor
    import torch
    p = capi.make_params(L.KERNEL_GI, 96, 64, max_ray_depth=3)
    outs = []
    for s in (sc, ref):
        t = torch.zeros((64, 96, 3), dtype=torch.float32, device="cuda:0")
        ctx.render_device(s, util.default_camera(), p, t.data_ptr(), sync=True)
        outs.append(t.cpu().numpy())
    util.assert_bit_equal(outs[0], outs[1], "%s lt_render_device" % name)
    ref.release()
    sc.release()


def test_refit_on_the_large_scene_paths():
    """lowered limits: the small scenes take the device-built threaded copies, k_flat_stream and the stack walk"""
    with capi.Context(0) as c:
        c.debug_limits(0, 0)
        for name in ("cornell_box", "cornell_box_lens"):
            sb = util.scene(name)
            sc = c.upload(sb)
            c.refit(sc, DEFORM[name](sb.prims))
            ref = fresh(c, sc, sb)
            assert not c.uses_traversal_tree(sc)
            check_renders(c, sc, ref, KERNELS, [0, L.FLAG_NO_THREADED, L.FLAG_NO_STREAM, L.FLAG_WAVEFRONT],
                          what="large-scene paths, " + name)
            ref.release()
            sc.release()


def test_refit_1m_mesh_renders_equal_fresh_upload(ctx, synth1m):
    sb, sc = synth1m
    ctx.refit(sc, sine(sb.prims))
    ref = fresh(ctx, sc, sb)
    cam = util.default_camera()
    for p in (capi.make_params(L.KERNEL_ACCUMULATOR, 1920, 1080),
              capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=4, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN)):
        ctx.accum_reset()
        got = ctx.render(sc, cam, p)
        ctx.accum_reset()
        want = ctx.render(ref, cam, p)
        util.assert_bit_equal(got, want, "1 M mesh, kernel %d" % p.kernel)
    ref.release()
    ctx.refit(sc, sb.prims)


def test_refit_cornell_matches_oracle(ctx):
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    ctx.refit(sc, translated(sb.prims))
    down = download(ctx, sc)
    moved = L.SceneBuffers(down.nodes, down.prims, sb.materials, down.lights)
    w, h = 96, 64
    cam = util.default_camera(0.02, 2)
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, w, h)
    oids, ohit, otuv, _ = O.primary_hits(2, moved, cam, w, h)
    assert (ids == oids).all() and (hit == ohit).all()
    assert tuv.view(np.uint32).tobytes() == otuv.view(np.uint32).tobytes()
    for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_CUSTOM_BARY):
        util.assert_bit_equal(ctx.render(sc, cam, capi.make_params(kernel, w, h)), O.render(kernel, moved, cam, w, h),
                              "deformed Cornell box, kernel %d vs oracle" % kernel)
    sc.release()


def test_refit_views_and_plugin_equal_fresh_upload(ctx):
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    ctx.refit(sc, translated(sb.prims))
    ref = fresh(ctx, sc, sb)
    cams = np.concatenate([L.make_camera(x, 2.5, z, yaw, fc)
                           for x, z, yaw, fc in ((0, -50, 0, 0), (1.5, -45, 0.05, 3), (-2, -55, -0.04, 7),
                                                 (0.5, -48, 0.02, 1))])
    p = capi.make_params(L.KERNEL_GI, 96, 64, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
    util.assert_bit_equal(ctx.render_views(sc, cams, p), ctx.render_views(ref, cams, p), "4 views")
    pid = ctx.plugin_load(GI_PLUGIN)
    pp = capi.make_params(0, 96, 64, frames=3, accum_mode=L.ACCUM_RUNNING_MEAN)
    pp.block_x, pp.block_y = 8, 8
    ctx.accum_reset()
    got = ctx.render_plugin_frames(sc, util.default_camera(0.02), pid, pp)
    ctx.accum_reset()
    want = ctx.render_plugin_frames(ref, util.default_camera(0.02), pid, pp)
    util.assert_bit_equal(got, want, "gi_plugin.cu frames")
    ref.release()
    sc.release()


def test_refit_round_trip(ctx):
    sb = util.scene("cornell_box_lens")
    sc = ctx.upload(sb)
    p = capi.make_params(L.KERNEL_GI, 96, 64, max_ray_depth=3, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
    cam = util.default_camera(0.02)
    ctx.accum_reset()
    before = ctx.render(sc, cam, p)
    ctx.refit(sc, scaled(sb.prims))
    ctx.accum_reset()
    moved = ctx.render(sc, cam, p)
    assert (moved != before).any()
    ctx.refit(sc, sb.prims)
    ctx.accum_reset()
    util.assert_bit_equal(ctx.render(sc, cam, p), before, "round trip")
    down = download(ctx, sc)
    assert down.nodes.tobytes() == restate_refit(sb.nodes, sb.prims).tobytes()
    # the host builder's inner boxes may hold the other zero (tests/test_scene_refit.py); every other bit is restored
    assert positive_zeros(down.nodes).tobytes() == positive_zeros(sb.nodes).tobytes()
    assert down.prims.tobytes() == sb.prims.tobytes()
    sc.release()


def test_repeated_refits_allocate_nothing(ctx):
    """the device memory the scene holds, counted by the library at each of its allocations: the first refit adds its
    parent links and scratch (and room for the largest pruned copies), later ones nothing"""
    for name in ("cornell_box_lens", "cornell_box"):
        sb = util.scene(name)
        sc = ctx.upload(sb)
        uploaded = ctx.scene_bytes(sc)
        assert uploaded > 0
        ctx.refit(sc, sb.prims)
        held = ctx.scene_bytes(sc)
        assert held > uploaded
        for k in range(50):
            ctx.refit(sc, sine(scaled(sb.prims, 1.0 + 0.004 * k), 0.05, 0.3 * k) if k % 2 else sb.prims)
            assert ctx.scene_bytes(sc) == held, "%s, refit %d" % (name, k)
        sc.release()


def test_rejected_first_refit_then_a_valid_one(ctx):
    """a scene whose first refit call is rejected derives its parent links and ranks on the next one"""
    import torch
    sb = util.scene("cornell_box_lens")
    prims = scaled(sb.prims)
    nan = prims.copy()
    nan["a"][3, 0] = np.nan
    bad_mat = prims.copy()
    bad_mat["mat"][2] = len(sb.materials)
    for form in ("device", "host"):
        for bad in (nan, bad_mat):
            sc = ctx.upload(sb)
            if form == "device":
                t = torch.from_numpy(bad.view(np.uint8).copy()).to("cuda:0")
                rc = ctx.lib.lt_scene_refit_device(ctx.h, sc.h, C.c_void_p(t.data_ptr()), bad.nbytes)
            else:
                rc = ctx.lib.lt_scene_refit(ctx.h, sc.h, bad.ctypes.data, bad.nbytes)
            assert rc == capi.ERR_INVALID
            check_nodes(ctx, sc, sb.nodes, prims, "valid refit after a rejected first %s refit" % form)
            ref = fresh(ctx, sc, sb)
            check_renders(ctx, sc, ref, [L.KERNEL_BASIC_CU, L.KERNEL_GI], [0, L.FLAG_NO_THREADED],
                          what="after a rejected first %s refit" % form)
            ref.release()
            sc.release()


def test_leaf_range_past_the_primitive_buffer_is_rejected(ctx):
    """lt_scene_upload checks a leaf's first primitive only; a refit reads them all, so it refuses such a scene"""
    import torch
    sb = util.scene("cornell_box")
    nodes = sb.nodes.copy()
    last = np.nonzero((nodes["count"] > 0) & (nodes["offset"] == len(sb.prims) - 1))[0]
    assert len(last) == 1
    nodes["count"][last[0]] = 2
    sc = ctx.upload(L.SceneBuffers(nodes, sb.prims, sb.materials, sb.lights))
    before = image(ctx, sc)
    prims = translated(sb.prims)
    t = torch.from_numpy(prims.view(np.uint8).copy()).to("cuda:0")
    for _ in range(2):
        assert ctx.lib.lt_scene_refit(ctx.h, sc.h, prims.ctypes.data, prims.nbytes) == capi.ERR_INVALID
        assert b"run past" in ctx.lib.lt_last_error(ctx.h)
        assert ctx.lib.lt_scene_refit_device(ctx.h, sc.h, C.c_void_p(t.data_ptr()), prims.nbytes) == capi.ERR_INVALID
    util.assert_bit_equal(image(ctx, sc), before, "after refused refits")
    down = download(ctx, sc)
    assert down.nodes.tobytes() == nodes.tobytes() and down.prims.tobytes() == sb.prims.tobytes()
    sc.release()


def image(ctx, sc):
    ctx.accum_reset()
    return ctx.render(sc, util.default_camera(0.02), capi.make_params(L.KERNEL_GI, 64, 48, max_ray_depth=3))


def test_rejected_inputs_leave_the_scene(ctx):
    import torch
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    ctx.refit(sc, translated(sb.prims))
    before, nodes = image(ctx, sc), download(ctx, sc).nodes.tobytes()
    bad = []
    wrong_mat = translated(sb.prims)
    wrong_mat["mat"][5] = len(sb.materials)
    bad.append(wrong_mat)
    neg_mat = translated(sb.prims)
    neg_mat["mat"][0] = -1
    bad.append(neg_mat)
    for k, v in (("a", np.nan), ("b", np.inf), ("c", -np.inf)):
        x = sb.prims.copy()
        x[k][7, 1] = v
        bad.append(x)
    lib = ctx.lib
    for prims in bad:
        assert lib.lt_scene_refit(ctx.h, sc.h, prims.ctypes.data, prims.nbytes) == capi.ERR_INVALID
        t = torch.from_numpy(prims.view(np.uint8).copy()).to("cuda:0")
        assert lib.lt_scene_refit_device(ctx.h, sc.h, C.c_void_p(t.data_ptr()), prims.nbytes) == capi.ERR_INVALID
    good = sb.prims
    t = torch.from_numpy(good.view(np.uint8).copy()).to("cuda:0")
    for n in (good.nbytes - 76, good.nbytes + 76, 0):
        assert lib.lt_scene_refit(ctx.h, sc.h, good.ctypes.data, n) == capi.ERR_INVALID
        assert lib.lt_scene_refit_device(ctx.h, sc.h, C.c_void_p(t.data_ptr()), n) == capi.ERR_INVALID
    assert lib.lt_scene_refit(ctx.h, None, good.ctypes.data, good.nbytes) == capi.ERR_INVALID
    assert lib.lt_scene_refit(ctx.h, sc.h, None, good.nbytes) == capi.ERR_INVALID
    assert lib.lt_scene_refit_device(ctx.h, sc.h, None, good.nbytes) == capi.ERR_INVALID
    # host memory is not device memory
    assert lib.lt_scene_refit_device(ctx.h, sc.h, good.ctypes.data, good.nbytes) == capi.ERR_INVALID
    # device memory that is not 4-byte aligned
    odd = torch.zeros(good.nbytes + 4, dtype=torch.uint8, device="cuda:0")
    for off in (1, 2, 3):
        assert lib.lt_scene_refit_device(ctx.h, sc.h, C.c_void_p(odd.data_ptr() + off), good.nbytes) == capi.ERR_INVALID
        assert b"aligned" in lib.lt_last_error(ctx.h)
    util.assert_bit_equal(image(ctx, sc), before, "after rejected refits")
    assert download(ctx, sc).nodes.tobytes() == nodes
    sc.release()


def test_device_form_from_a_torch_tensor(ctx):
    import torch
    sb = util.scene("cornell_box_lens")
    prims = scaled(sb.prims)
    a, b = ctx.upload(sb), ctx.upload(sb)
    ctx.refit(a, prims)
    t = torch.from_numpy(prims.view(np.uint8).copy()).to("cuda:0")
    ctx.refit_device(b, t.data_ptr(), prims.nbytes)
    assert ctx.stats().upload_ms > 0.0
    assert download(ctx, a).nodes.tobytes() == download(ctx, b).nodes.tobytes()
    assert download(ctx, b).prims.tobytes() == prims.tobytes()
    util.assert_bit_equal(image(ctx, a), image(ctx, b), "device form")
    a.release()
    b.release()


def test_refit_every_device_copy():
    for n in util.group_sizes():
        refit_every_device_copy(n)


def refit_every_device_copy(n):
    sb = util.scene("cornell_box")
    prims = translated(sb.prims)
    with capi.Context(0) as one, util.device_group(n) as many:
        a, m = one.upload(sb), many.upload(sb)
        one.refit(a, prims)
        many.refit(m, prims)
        assert many.lib.lt_scene_refit_device(many.h, m.h, C.c_void_p(1), prims.nbytes) == -4  # LT_ERR_UNSUPPORTED
        p = capi.make_params(L.KERNEL_BASIC_CU, 96, 64, split_mode=L.SPLIT_TILES)
        cam = util.default_camera(0.02)
        # every device renders rows of the image from its own copy
        util.assert_bit_equal(many.render(m, cam, p), one.render(a, cam, p), "multi-GPU refit, tile split")
        a.release()
        m.release()

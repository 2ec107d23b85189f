"""GPU parity tests added in round 2: the persistent pixel-dealing kernels, odd image sizes, deep trees, deep
bounce caps, and the BASELINE.json configurations AT THEIR FULL SIZES (1 M-triangle mesh at 1080p and 4K, the
custom kernel at 1080p x 16 through RendererOpenCL::render) against the CPU oracle on the same buffers."""
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L
from test_gpu_parity import PIPES, assert_images_match

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def synth1m(ctx, tmp_path_factory):
    """BASELINE.json configs[2]: the synthetic 1 M-triangle mesh (grid 707 -> 999 710 triangles, 1 999 419 nodes)."""
    p = str(tmp_path_factory.mktemp("synth") / "synth707.obj")
    host.write_synthetic_scene(p, 707, 0x5EED)
    sb = host.load_scene_buffers(p)
    sc = ctx.upload(sb)
    yield sb, sc
    sc.release()


def chain_scene(n):
    """A maximally unbalanced tree over n stacked triangles: inner node 2k has leaf 2k+1 and inner node 2k+2 as
    children, so the traversal stack needs n - 1 levels (validate_tree) -- beyond 40 the culled mode asks for more
    than 48 KB of dynamic shared memory per block."""
    prims = np.zeros(n, L.PRIM)
    nodes = np.zeros(2 * n - 1, L.NODE)
    for i in range(n):
        z = 1.0 + 0.25 * i
        x = -2.0 + 4.0 * (i % 7) / 7.0
        prims["a"][i] = (x - 1.5, 1.0, z)
        prims["b"][i] = (x + 1.5, 1.0, z)
        prims["c"][i] = (x, 4.0, z + 0.1)
        for k in ("na", "nb", "nc"):
            prims[k][i] = (0, 0, -1)
        prims["mat"][i] = i % 3
    lo = np.minimum(np.minimum(prims["a"], prims["b"]), prims["c"])
    hi = np.maximum(np.maximum(prims["a"], prims["b"]), prims["c"])
    for i in range(n - 1):
        inner, leaf = 2 * i, 2 * i + 1
        nodes["min"][inner] = lo[i:].min(axis=0)
        nodes["max"][inner] = hi[i:].max(axis=0)
        nodes["offset"][inner] = 2 * i + 2
        nodes["count"][inner] = 0
        nodes["axis"][inner] = 2
        nodes["min"][leaf], nodes["max"][leaf] = lo[i], hi[i]
        nodes["offset"][leaf] = i
        nodes["count"][leaf] = 1
    last = 2 * n - 2
    nodes["min"][last], nodes["max"][last] = lo[n - 1], hi[n - 1]
    nodes["offset"][last] = n - 1
    nodes["count"][last] = 1
    mats = np.zeros(3, L.MATERIAL)
    mats["diffuse"] = [(0.9, 0.2, 0.2), (0.2, 0.9, 0.2), (0.2, 0.2, 0.9)]
    mats["ior"] = 1.0
    mats["dissolve"] = 1.0
    mats["emission"][2] = (1, 1, 1)
    lights = np.zeros(1, L.LIGHTS)
    em = [i for i in range(n) if i % 3 == 2][:4]
    lights["count"] = len(em)
    lights["prims"][0][:len(em)] = em
    return L.SceneBuffers(nodes, prims, mats, lights)


# ---------------------------------------------------------------------------------------------------------------
# ADVICE round 1: odd path counts, deep bounce caps, deep trees, unreachable nodes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [(101, 75), (101, 101), (33, 17), (1, 1)])
@pytest.mark.parametrize("frames", [1, 3])
def test_odd_image_sizes_in_the_wavefront_pipeline(ctx, size, frames):
    """An odd number of paths per batch once left the second batch workspace and the primary records 8 bytes off a
    16-byte boundary (misaligned float4 accesses).  All schedules, one and two streams, against the oracle."""
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    w, h = size
    acc = np.zeros((h, w, 3), np.float32)
    for f in range(frames):
        O.accumulate(acc, O.render(L.KERNEL_GI, sb, util.default_camera(0.0, f), w, h, max_ray_depth=3, threads=0), f)
    for flags in (L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_SERIAL, L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED,
                  L.FLAG_MEGAKERNEL):
        ctx.accum_reset()
        got = ctx.render(sc, util.default_camera(0.0, 0),
                         capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, frames=frames,
                                          accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags))
        assert_images_match(got, acc, "odd size %dx%d x%d flags %d" % (w, h, frames, flags), max_outliers=3)
    sc.release()


def test_bounce_caps_beyond_the_wavefront_depth_field(ctx):
    """The wavefront queue entry carries the bounce depth in 5 bits: max_ray_depth > 32 must not wrap.  The default
    schedule keeps such launches on the megakernel; forcing the wavefront is a reported error."""
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    cam = util.default_camera(0.0, 3)
    w, h = 96, 64
    want = O.render(L.KERNEL_GI, sb, cam, w, h, max_ray_depth=40, threads=0)
    got = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=40))
    assert_images_match(got, want, "max_ray_depth 40, default schedule", max_outliers=3)
    # enough paths for the wavefront to be the default choice: still correct (falls back to the megakernel)
    ctx.accum_reset()
    big = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=33, frames=5,
                                               accum_mode=L.ACCUM_RUNNING_MEAN, flags=0)).copy()
    ctx.accum_reset()
    mega = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=33, frames=5,
                                                accum_mode=L.ACCUM_RUNNING_MEAN, flags=L.FLAG_MEGAKERNEL)).copy()
    util.assert_bit_equal(big, mega, "depth 33: default schedule vs megakernel")
    with pytest.raises(capi.LtError):
        ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=33, flags=L.FLAG_WAVEFRONT))
    at32 = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=32, flags=L.FLAG_WAVEFRONT))
    assert_images_match(at32, O.render(L.KERNEL_GI, sb, cam, w, h, max_ray_depth=32, threads=0), "depth 32 wavefront",
                        max_outliers=3)
    sc.release()


@pytest.mark.parametrize("n", [45, 62])
def test_deep_tree_in_every_mode(ctx, n):
    """Stack depth 44 / 61: the culled mode needs (2 * depth + 16) * 512 bytes of dynamic shared memory (> 48 KB:
    an opt-in per kernel).  Exact, culled, stack and threaded traversal all equal the oracle."""
    sb = chain_scene(n)
    sc = ctx.upload(sb)
    assert ctx.download(sc)[1] == n - 1
    cam = L.make_camera(0.0, 2.5, -20.0, 0.0, 1)
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 160, 120)
    oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, 160, 120)
    assert hit.sum() > 100
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv)
    cids, chit, ctuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 160, 120, flags=L.FLAG_CULL)
    np.testing.assert_array_equal(cids, oids)
    util.assert_bit_equal(ctuv, otuv)
    for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_ACCUMULATOR, L.KERNEL_GI):
        want = O.render(kernel, sb, cam, 160, 120, max_ray_depth=3, threads=0)
        for flags in (0, L.FLAG_NO_STREAM, L.FLAG_CULL, L.FLAG_NO_THREADED, L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED,
                      L.FLAG_WAVEFRONT | L.FLAG_CULL, L.FLAG_MEGAKERNEL):
            if kernel == L.KERNEL_BASIC_CU and flags & (L.FLAG_WAVEFRONT | L.FLAG_MEGAKERNEL):
                continue
            got = ctx.render(sc, cam, capi.make_params(kernel, 160, 120, max_ray_depth=3, flags=flags))
            assert_images_match(got, want, "chain %d kernel %d flags %d" % (n, kernel, flags), max_outliers=3)
    sc.release()


def test_unreachable_nodes_are_rejected(ctx):
    sb = util.scene("cornell_box")
    nodes = np.concatenate([sb.nodes, sb.nodes[-1:]])  # one array entry no parent points at
    with pytest.raises(capi.LtError) as e:
        ctx.upload(L.SceneBuffers(nodes, sb.prims, sb.materials, sb.lights))
    assert "reachable" in str(e.value)


# ---------------------------------------------------------------------------------------------------------------
# persistent pixel-dealing kernels == one thread per pixel
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens"])
@pytest.mark.parametrize("size", [(1920, 1080), (257, 130), (7, 3), (1, 1)])
def test_streamed_flat_kernel_equals_one_thread_per_pixel(name, size):
    """k_flat_stream (persistent warps that fetch 8x4 tiles; the default on large scenes, forced here on the small
    ones through a context whose stream_min_nodes limit is 0) == k_flat == the oracle, including the lens path and the
    frame combiner."""
    ctx = capi.Context(0)
    ctx.debug_limits(threaded_max_nodes=65536, stream_min_nodes=0)
    sb = util.scene(name)
    sc = ctx.upload(sb)
    w, h = size
    for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY):
        for yaw in (0.0, 0.06):
            cam = util.default_camera(yaw)
            imgs = [ctx.render(sc, cam, capi.make_params(kernel, w, h, flags=f)).copy()
                    for f in (0, L.FLAG_NO_STREAM, L.FLAG_NO_THREADED, L.FLAG_NO_THREADED | L.FLAG_NO_STREAM)]
            for k in range(1, 4):
                util.assert_bit_equal(imgs[0], imgs[k], "%s kernel %d: variant %d vs streamed" % (name, kernel, k))
            if w * h <= 257 * 130:
                util.assert_bit_equal(imgs[0], O.render(kernel, sb, cam, w, h), "%s kernel %d vs oracle" % (name, kernel))
    # frames through the frame combiner, depth 4
    cam = util.default_camera()
    a = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h, depth=4, frames=5, accum_mode=L.ACCUM_RUNNING_MEAN))
    b = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h, depth=4, frames=5, accum_mode=L.ACCUM_RUNNING_MEAN,
                                             flags=L.FLAG_NO_STREAM))
    util.assert_bit_equal(a[..., :3], b[..., :3], "running mean of a deterministic kernel")
    sc.release()
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# BASELINE.json configurations at their full sizes
# ---------------------------------------------------------------------------------------------------------------
def test_synth1m_primary_hits_full_frame_bit_exact(ctx, synth1m):
    """configs[2] mesh, 1920x1080: primitiveIndex / hitType / t / u / v of every camera ray == the oracle on the
    same buffers, and the flat pipeline (persistent and one-thread-per-pixel, exact and culled) agrees."""
    sb, sc = synth1m
    cam = util.default_camera()
    w, h = 1920, 1080
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, w, h)
    oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, w, h)
    np.testing.assert_array_equal(hit, ohit)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv, "1 M triangles: t,u,v at 1080p")
    assert len(np.unique(ids)) > 50000  # the frame really sees the mesh
    want = O.render(L.KERNEL_BASIC_CU, sb, cam, w, h)
    for flags in (0, L.FLAG_NO_STREAM, L.FLAG_CULL):
        got = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h, flags=flags))
        util.assert_bit_equal(got, want, "1 M triangles: basic.cu image, flags %d" % flags)


def test_synth1m_shadow_and_gi_all_schedules(ctx, synth1m):
    """configs[2] (primary + shadow, 1080p, 1 spp) full frame against the oracle; GI 4 bounces: bands against the
    oracle and all schedules bit-identical over the whole frame."""
    sb, sc = synth1m
    w, h = 1920, 1080
    cam = util.default_camera(0.0, 0)
    want = O.render(L.KERNEL_ACCUMULATOR, sb, cam, w, h, threads=0)
    imgs = []
    for flags in (0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT):
        got = ctx.render(sc, cam, capi.make_params(L.KERNEL_ACCUMULATOR, w, h, flags=flags)).copy()
        assert_images_match(got, want, "1 M triangles: primary + shadow, flags %d" % flags, max_outliers=8)
        imgs.append(got)
    util.assert_bit_equal(imgs[0], imgs[1], "default vs megakernel")
    util.assert_bit_equal(imgs[0], imgs[2], "megakernel vs wavefront")
    cam = util.default_camera(0.0, 5)
    gi = [ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, flags=f)).copy()
          for f in (0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_SERIAL)]
    for k in range(1, 4):
        util.assert_bit_equal(gi[0], gi[k], "GI on 1 M triangles: schedule %d vs default" % k)
    for rows in ((0, 8), (536, 552), (1072, 1080)):
        band = O.render(L.KERNEL_GI, sb, cam, w, h, max_ray_depth=4, rows=rows, threads=0)
        assert_images_match(gi[0][rows[0]:rows[1]], band[rows[0]:rows[1]], "GI rows %s" % (rows,), max_outliers=4)


def test_synth1m_4k_five_frames(ctx, synth1m):
    """3840x2160, 5 frames on the 1 M-triangle mesh: 8.3 M pixels per frame -> three frames per wavefront batch
    (path ids are 25 bits: at most four; five frames halved for two overlapped batches).  Whole frame: wavefront ==
    megakernel bit for bit; bands == the oracle's running mean of the same five frames."""
    sb, sc = synth1m
    w, h, frames = 3840, 2160, 5
    cam0 = util.default_camera(0.0, 0)
    p = dict(max_ray_depth=4, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN)
    ctx.accum_reset()
    wf = ctx.render(sc, cam0, capi.make_params(L.KERNEL_GI, w, h, flags=0, **p)).copy()
    assert ctx.stats().kernel_launches > 10  # the default schedule at this size is the wavefront pipeline
    ctx.accum_reset()
    mega = ctx.render(sc, cam0, capi.make_params(L.KERNEL_GI, w, h, flags=L.FLAG_MEGAKERNEL, **p)).copy()
    util.assert_bit_equal(wf, mega, "4K x 5 frames: wavefront vs megakernel")
    for rows in ((1000, 1012), (2148, 2160)):
        acc = np.zeros((h, w, 3), np.float32)
        for f in range(frames):
            O.accumulate(acc, O.render(L.KERNEL_GI, sb, util.default_camera(0.0, f), w, h, max_ray_depth=4, rows=rows,
                                       threads=0), f)
        assert_images_match(wf[rows[0]:rows[1]], acc[rows[0]:rows[1]], "4K rows %s" % (rows,), max_outliers=6)


def test_custom_kernel_config_full_size_through_renderer_opencl(root):
    """BASELINE.json configs[3]: the custom_kernel example's shading plug-in (custom_opencl.cl) on the Cornell OBJ,
    1920x1080, 16 accumulated frames, through RendererOpenCL::render with a RenderExtensionB200 -- against the
    oracle's running mean of 16 (identical) frames, every pixel."""
    cwd = os.getcwd()
    os.chdir(root)
    try:
        w, h = 1920, 1080
        model = host.Model("resources/models/cornell_box.obj")
        accel = host.AccelerationStructure(model)
        cam = host.Camera(0, 2.5, -50, 0)
        r = host.Renderer(host.PLATFORM_OPENCL)
        ext = host.make_extension(frames=16, accumulate=True)
        got = r.render("examples/custom_kernel/resources/kernels/custom_opencl.cl", w, h, accel, model, cam, ext=ext)
        sb = accel.buffers()
        one = O.render(L.KERNEL_CUSTOM_BARY, sb, util.default_camera(), w, h)
        acc = np.zeros_like(one)
        for f in range(16):
            O.accumulate(acc, one, f)
        util.assert_bit_equal(got, acc, "custom kernel 1080p x 16")
        assert (got.max(axis=-1) > 0).mean() > 0.2
        # the reference protocol: 16 render() calls of one frame each, frameCount incremented by the caller
        # (examples/global_illumination/src/main.cpp:296-325), accumulated on the host like accumulator.frag
        acc2 = np.zeros_like(one)
        for f in range(16):
            cam.set_frame_count(f)
            frame = r.render("examples/custom_kernel/resources/kernels/custom_opencl.cl", w, h, accel, model, cam)
            O.accumulate(acc2, frame, f)
        util.assert_bit_equal(acc2, acc, "custom kernel, 16 single-frame render() calls")
        r.close(); accel.close(); model.close(); cam.close()
    finally:
        os.chdir(cwd)


def test_sah_tree_on_the_gpu(ctx, tmp_path):
    """The opt-in binned-SAH tree (ACCELERATION_STRUCTURE_TYPE_SAH_B200): kernels == oracle on identical buffers (ids,
    t/u/v bit-exact, GI within the usual bound), in every schedule, on the Cornell box and an 80 k-triangle mesh."""
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 200, 0x5EED)
    for path in (os.path.join(util.MODELS, "cornell_box.obj"), p):
        sb = host.load_scene_buffers(path, host.AccelerationStructure.HOST_SAH)
        sc = ctx.upload(sb)
        cam = util.default_camera(0.0, 2)
        ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 320, 180)
        oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, 320, 180)
        np.testing.assert_array_equal(ids, oids)
        util.assert_bit_equal(tuv, otuv, "SAH tree: t,u,v")
        want = O.render(L.KERNEL_GI, sb, cam, 160, 90, max_ray_depth=4, threads=0)
        for pipe in [0] + PIPES:
            got = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 160, 90, max_ray_depth=4, flags=pipe))
            assert_images_match(got, want, "SAH tree GI, flags %d" % pipe, max_outliers=3)
        sc.release()


def test_device_built_threaded_copies():
    """Large trees get their eight threaded (skip-pointer) copies from a device kernel (k_build_threaded) and use them
    for coherent-ray launches.  A context whose threaded_max_nodes limit is 0 sends the small test scenes down that
    path too: deterministic and lighting kernels must still equal the oracle bit for bit, and the stack traversal."""
    ctx = capi.Context(0)
    ctx.debug_limits(threaded_max_nodes=0, stream_min_nodes=0)
    for name in ("cornell_box", "cornell_box_lens", "green_wall", "single"):
        sb = util.single_triangle_scene() if name == "single" else util.scene(name)
        sc = ctx.upload(sb)
        for yaw in (0.0, 0.05, -2.5):
            cam = util.default_camera(yaw, 2)
            for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_CUSTOM_BARY, L.KERNEL_ACCUMULATOR, L.KERNEL_LIGHTING25):
                w, h = (160, 100) if kernel != L.KERNEL_LIGHTING25 else (48, 32)
                mega = L.FLAG_MEGAKERNEL if kernel >= L.KERNEL_LIGHTING25 else 0
                got = ctx.render(sc, cam, capi.make_params(kernel, w, h, flags=mega))
                want = O.render(kernel, sb, cam, w, h, threads=0)
                bad = (got.view(np.uint32) != want.view(np.uint32)).any(axis=-1).sum()
                assert bad <= (3 if kernel >= L.KERNEL_LIGHTING25 else 0), (name, yaw, kernel, int(bad))
                stack = ctx.render(sc, cam, capi.make_params(kernel, w, h, flags=L.FLAG_NO_THREADED | mega))
                assert (got.view(np.uint32) == stack.view(np.uint32)).all(), (name, yaw, kernel)
        sc.release()
    ctx.close()

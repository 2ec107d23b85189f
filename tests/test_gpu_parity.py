"""GPU parity tests: the CUDA path, called through the C-ABI, against the CPU oracle on the same
buffers.  Bar: bit-exact for primitive ids / hit flags, and bit-exact FP32 for every deterministic
pass (tolerance only where the fp64 device sin/cos of the hash RNG may differ from libm in the last
place: at most a handful of pixels, each checked to 1e-4 relative)."""
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu

FLAVOUR = {L.KERNEL_BASIC_CU: 0, L.KERNEL_BASIC_CL: 1, L.KERNEL_CUSTOM_BARY: 1, L.KERNEL_LIGHTING25: 1,
           L.KERNEL_ACCUMULATOR: 2, L.KERNEL_GI25: 2, L.KERNEL_GI: 2}


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


_uploaded = {}


def gpu_scene(ctx, name):
    if name not in _uploaded:
        sb = {"single": util.single_triangle_scene, "single_light": lambda: util.single_triangle_scene(True),
              "multi_leaf": util.multi_prim_leaf_scene}.get(name, lambda: util.scene(name))()
        _uploaded[name] = (sb, ctx.upload(sb))
    return _uploaded[name]


def assert_images_match(got, want, what, max_outliers=0):
    """bit-exact, except for at most max_outliers pixels which must still agree to 1e-4 relative"""
    gb, wb = util.bits(got), util.bits(want)
    bad = (gb != wb).any(axis=-1)
    n = int(bad.sum())
    if n == 0:
        return
    assert n <= max_outliers, "%s: %d pixels differ bitwise (allowed %d)" % (what, n, max_outliers)
    np.testing.assert_allclose(got[bad], want[bad], rtol=1e-4, atol=1e-6, err_msg=what)


@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens", "single", "multi_leaf"])
@pytest.mark.parametrize("size", [(100, 100), (33, 17), (1, 1), (257, 130)])
@pytest.mark.parametrize("yaw", [0.0, 0.04, -0.07, -2.5])  # |yaw| < 0.1 keeps the model in view
def test_primary_hit_records_bit_exact(ctx, name, size, yaw):
    sb, sc = gpu_scene(ctx, name)
    cam = util.default_camera(yaw)
    w, h = size
    for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_GI):
        ids, hit, tuv = ctx.primary_hits(sc, cam, kernel, w, h)
        oids, ohit, otuv, _ = O.primary_hits(FLAVOUR[kernel], sb, cam, w, h)
        np.testing.assert_array_equal(hit, ohit)
        np.testing.assert_array_equal(ids, oids)
        util.assert_bit_equal(tuv, otuv, "%s t,u,v" % name)


@pytest.mark.parametrize("kernel", [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY])
@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens", "single"])
@pytest.mark.parametrize("yaw", [0.0, -0.05, 0.2])
def test_deterministic_kernels_bit_exact(ctx, kernel, name, yaw):
    sb, sc = gpu_scene(ctx, name)
    cam = util.default_camera(yaw)
    for w, h, mode in ((100, 100, 0), (161, 75, 1)):
        got = ctx.render(sc, cam, capi.make_params(kernel, w, h, kernel_mode=mode))
        want = O.render(kernel, sb, cam, w, h, kernel_mode=mode)
        util.assert_bit_equal(got, want, "%s kernel %d" % (name, kernel))


def test_reference_known_answer_on_gpu(ctx):
    # tests/cuda_renderer_test.cc:182-225
    sb, sc = gpu_scene(ctx, "green_wall")
    flat = ctx.render(sc, util.default_camera(), capi.make_params(L.KERNEL_BASIC_CU, 100, 100)).reshape(-1)
    for x in range(0, 100 * 100, 8 * 3):
        assert flat[x] == 0.0 and flat[x + 1] == 1.0 and flat[x + 2] == 0.0


# the schedules of the stochastic kernels (identical output): persistent megakernel, wavefront with the stackless
# threaded traversal (small scenes), wavefront with the stack traversal
PIPES = [L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED]


@pytest.mark.parametrize("pipe", PIPES)
@pytest.mark.parametrize("kernel,depth", [(L.KERNEL_ACCUMULATOR, 0), (L.KERNEL_GI, 4), (L.KERNEL_GI, 16),
                                          (L.KERNEL_GI, 1)])
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "single_light"])
@pytest.mark.parametrize("frame", [0, 1, 7, 63])
def test_stochastic_single_sample(ctx, pipe, kernel, depth, name, frame):
    sb, sc = gpu_scene(ctx, name)
    cam = util.default_camera(0.0, frame)
    w, h = 128, 96
    got = ctx.render(sc, cam, capi.make_params(kernel, w, h, max_ray_depth=depth, flags=pipe))
    want = O.render(kernel, sb, cam, w, h, max_ray_depth=depth if depth else 16, threads=0)
    assert np.isfinite(got).all()
    assert_images_match(got, want, "kernel %d frame %d" % (kernel, frame), max_outliers=3)


@pytest.mark.parametrize("pipe", PIPES)
@pytest.mark.parametrize("kernel", [L.KERNEL_LIGHTING25, L.KERNEL_GI25])
@pytest.mark.parametrize("mode", [0, 1])
def test_blend25_kernels(ctx, pipe, kernel, mode):
    sb, sc = gpu_scene(ctx, "cornell_box")
    cam = util.default_camera(0.05, 2)
    got = ctx.render(sc, cam, capi.make_params(kernel, 64, 48, kernel_mode=mode, max_ray_depth=3, flags=pipe))
    want = O.render(kernel, sb, cam, 64, 48, kernel_mode=mode, max_ray_depth=3, threads=0)
    assert_images_match(got, want, "blend25 kernel %d" % kernel, max_outliers=3)


@pytest.mark.parametrize("pipe", PIPES)
def test_running_mean_matches_frame_by_frame_protocol(ctx, pipe):
    """examples/global_illumination/src/main.cpp:296-325: one sample per frame, frameCount = 0,1,2..,
    running mean.  One multi-frame launch == the oracle rendering frame by frame and accumulating."""
    sb, sc = gpu_scene(ctx, "cornell_box")
    w, h, frames = 96, 64, 6
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                         flags=pipe)
    ctx.accum_reset()
    got = ctx.render(sc, util.default_camera(0.0, 0), p)
    acc = np.zeros((h, w, 3), np.float32)
    for f in range(frames):
        O.accumulate(acc, O.render(L.KERNEL_GI, sb, util.default_camera(0.0, f), w, h, max_ray_depth=4, threads=0), f)
    assert_images_match(got, acc, "running mean", max_outliers=3)
    # the same through successive single-frame calls sharing the context accumulator
    ctx.accum_reset()
    for f in range(frames):
        p1 = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=1, accum_mode=L.ACCUM_RUNNING_MEAN,
                              flags=pipe)
        step = ctx.render(sc, util.default_camera(0.0, f), p1)
    util.assert_bit_equal(step, got, "multi-frame launch vs frame-by-frame launches")


def test_accumulating_a_deterministic_kernel(ctx):
    # BASELINE config 4: custom kernel, 16 accumulated frames
    sb, sc = gpu_scene(ctx, "cornell_box")
    w, h = 120, 80
    p = capi.make_params(L.KERNEL_CUSTOM_BARY, w, h, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN)
    got = ctx.render(sc, util.default_camera(), p)
    one = O.render(L.KERNEL_CUSTOM_BARY, sb, util.default_camera(), w, h)
    acc = np.zeros_like(one)
    for f in range(16):
        O.accumulate(acc, one, f)
    util.assert_bit_equal(got, acc)
    np.testing.assert_allclose(got, one, rtol=1e-6, atol=1e-7)


def test_wavefront_batches_equal_one_batch(ctx, monkeypatch):
    """frames split over several wavefront batches (workspace cap) == megakernel, bit for bit"""
    sb, sc = gpu_scene(ctx, "cornell_box")
    w, h, frames = 64, 48, 7
    cam = util.default_camera(0.0, 3)
    ctx.accum_reset()
    a = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, frames=frames,
                                             accum_mode=L.ACCUM_RUNNING_MEAN, flags=L.FLAG_MEGAKERNEL))
    ctx.accum_reset()
    b = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, frames=frames,
                                             accum_mode=L.ACCUM_RUNNING_MEAN, flags=L.FLAG_WAVEFRONT))
    util.assert_bit_equal(a, b, "wavefront vs megakernel")


def test_weighted_sum_split_equals_mean(ctx):
    # sample split across G "ranks": rank g renders frames g, g+G, .. weighted 1/N; the sum is the mean
    sb, sc = gpu_scene(ctx, "cornell_box")
    w, h, n, g = 64, 64, 8, 4
    total = np.zeros((h, w, 3), np.float64)
    for r in range(g):
        ctx.accum_reset()
        p = capi.make_params(L.KERNEL_ACCUMULATOR, w, h, frames=n // g, frame_stride=g,
                             accum_mode=L.ACCUM_WEIGHTED_SUM, accum_weight=1.0 / n)
        total += ctx.render(sc, util.default_camera(0.0, r), p)
    ctx.accum_reset()
    mean = ctx.render(sc, util.default_camera(0.0, 0),
                      capi.make_params(L.KERNEL_ACCUMULATOR, w, h, frames=n, accum_mode=L.ACCUM_RUNNING_MEAN))
    np.testing.assert_allclose(total, mean, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("pipe", PIPES)
def test_stats_count_the_reference_traversal(ctx, pipe):
    for name, kernel, depth in (("cornell_box", L.KERNEL_BASIC_CU, 0), ("cornell_box_lens", L.KERNEL_BASIC_CU, 0),
                                ("cornell_box", L.KERNEL_GI, 4), ("multi_leaf", L.KERNEL_BASIC_CU, 0)):
        sb, sc = gpu_scene(ctx, name)
        cam = util.default_camera(0.0, 1)
        ctx.render(sc, cam, capi.make_params(kernel, 96, 96, max_ray_depth=depth, flags=L.FLAG_STATS | pipe))
        st = ctx.stats()
        _, ost = O.render(kernel, sb, cam, 96, 96, max_ray_depth=depth if depth else 16, with_stats=True, threads=0)
        assert (st.rays, st.node_tests, st.tri_tests) == (ost.rays, ost.nodeTests, ost.triTests), name


def test_stats_mode_does_not_change_the_image(ctx):
    sb, sc = gpu_scene(ctx, "cornell_box")
    cam = util.default_camera(0.0, 5)
    a = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 80, 60, max_ray_depth=4))
    b = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 80, 60, max_ray_depth=4, flags=L.FLAG_STATS))
    util.assert_bit_equal(a, b)


@pytest.mark.parametrize("kernel,depth,frames", [(L.KERNEL_GI, 4, 7), (L.KERNEL_ACCUMULATOR, 0, 6), (L.KERNEL_GI25, 2, 2)])
def test_overlapped_batches_equal_one_stream(ctx, kernel, depth, frames):
    """Consecutive batches of the wavefront pipeline run on two streams (a trace kernel beside the other batch's
    shade kernel); the frame combiner is still applied in frame order, so the image is the one-stream image."""
    sb, sc = gpu_scene(ctx, "cornell_box")
    cam = util.default_camera(0.0, 0)
    w, h = (160, 120) if kernel != L.KERNEL_GI25 else (64, 48)
    imgs = []
    for flags in (L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_SERIAL, L.FLAG_MEGAKERNEL):
        ctx.accum_reset()
        imgs.append(ctx.render(sc, cam, capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames,
                                                         accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)).copy())
    util.assert_bit_equal(imgs[0], imgs[1], "two streams vs one stream")
    util.assert_bit_equal(imgs[0], imgs[2], "wavefront vs megakernel")


def test_shared_primary_hits_equal_per_frame_tracing(ctx):
    """The wavefront pipeline traces the camera ray of a pixel once per launch, starts every frame's path from that
    record (the ray is the same in every frame) and gives paths only to the pixels whose camera ray hits a surface
    (black / white pixels are constant).  Its stats launch traces the camera ray per frame and gives every pixel a
    path, and the megakernel traces it per frame as the reference does: all three images are the same."""
    sb, sc = gpu_scene(ctx, "cornell_box_lens")
    cam = util.default_camera(0.01, 2)

    def gi(flags):
        ctx.accum_reset()
        return ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 200, 150, max_ray_depth=3, frames=5,
                                                    accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)).copy()

    shared = gi(L.FLAG_WAVEFRONT)
    util.assert_bit_equal(shared, gi(L.FLAG_WAVEFRONT | L.FLAG_STATS),
                          "shared primary hits + alive list vs per-frame tracing for every pixel (stats launch)")
    util.assert_bit_equal(shared, gi(L.FLAG_MEGAKERNEL), "shared primary hits + alive list vs megakernel")
    lit = capi.make_params(L.KERNEL_ACCUMULATOR, 200, 150, frames=5, accum_mode=L.ACCUM_RUNNING_MEAN, flags=L.FLAG_WAVEFRONT)
    mega = capi.make_params(L.KERNEL_ACCUMULATOR, 200, 150, frames=5, accum_mode=L.ACCUM_RUNNING_MEAN, flags=L.FLAG_MEGAKERNEL)
    ctx.accum_reset()
    a = ctx.render(sc, cam, lit).copy()
    ctx.accum_reset()
    b = ctx.render(sc, cam, mega).copy()
    util.assert_bit_equal(a, b, "accumulator kernel (white light pixels): wavefront with alive list vs megakernel")
    assert len(np.unique(a.reshape(-1, 3), axis=0)) > 3  # black, the light's constant colour, shaded surfaces


def test_device_rng_matches_the_oracle(ctx):
    """random() (basic_lighting.cl:64-67) on the device -- exact fmod, the CUDA library's fp64 sin -- against the
    restatement (libm): 400 000 draws over the film positions and seeds a 1080p 64-spp step uses.  The two sines
    may differ in the last place of the double, which flips the FP32 rounding of sin * 43758.5453 with probability
    ~1e-9 per draw: at most 2 of the draws may differ, by one FP32 step of that product.  (A purpose-built sin for
    |y| < pi -- 20 instructions instead of ~150 -- was measured and did not shorten the shade kernel, which waits on
    memory, so the library function stays.)"""
    rng = np.random.default_rng(11)
    n = 400000
    px = rng.integers(0, 1920, n)
    py = rng.integers(0, 1080, n)
    fx = (px.astype(np.float32) / np.float32(1920) + np.float32(-0.5)).astype(np.float32)
    fy = (py.astype(np.float32) / np.float32(1080) + np.float32(-0.5)).astype(np.float32)
    seed = rng.integers(0, 64 * 32 + 40, n).astype(np.float32)
    seed[::97] = rng.integers(0, 1 << 24, len(seed[::97])).astype(np.float32)  # large frame counts
    dev = ctx.debug_random(fx, fy, seed)
    host = np.array([O.random(float(a), float(b), float(c)) for a, b, c in zip(fx, fy, seed)], dtype=np.float32)
    bad = dev != host
    assert bad.sum() <= 2, (int(bad.sum()), dev[bad][:4], host[bad][:4])
    assert np.abs(dev[bad] - host[bad]).max(initial=0.0) <= 2.0 ** -8 + 1e-7
    assert dev.min() >= 0.0 and dev.max() <= 1.0


def test_leaf_fifo_capacity_on_a_deep_tree(ctx, tmp_path):
    """Regression: one step of the stack traversal can record three leaves (near, far, and one popped behind
    them); with room for only two the FIFO overwrote its oldest entry -- one pixel of this 1080p frame.  All
    schedules must agree, and agree with the oracle on the rows around that pixel."""
    from lens_trace_b200 import host
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 96, 0x5EED)
    sb = host.load_scene_buffers(p)
    sc = ctx.upload(sb)
    cam = util.default_camera(0.0, 8)
    imgs = [ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=4, flags=pipe)).copy()
            for pipe in PIPES]
    sc.release()
    util.assert_bit_equal(imgs[1], imgs[0], "wavefront threaded vs megakernel")
    util.assert_bit_equal(imgs[2], imgs[0], "wavefront stack vs megakernel")
    want = O.render(L.KERNEL_GI, sb, cam, 1920, 1080, max_ray_depth=4, rows=(540, 548), threads=0)
    assert_images_match(imgs[2][540:548], want[540:548], "rows 540..547 vs oracle", max_outliers=3)


def test_synthetic_mesh_parity(ctx, tmp_path):
    from lens_trace_b200 import host
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 96, 0x5EED)  # 18 444 triangles
    sb = host.load_scene_buffers(p)
    sc = ctx.upload(sb)
    cam = util.default_camera()
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 200, 120)
    oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, 200, 120)
    np.testing.assert_array_equal(hit, ohit)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv)
    want = O.render(L.KERNEL_GI, sb, util.default_camera(0.0, 3), 160, 90, max_ray_depth=4, threads=0)
    for pipe in [0] + PIPES:  # default choice, megakernel, wavefront threaded (36 887 nodes), wavefront stack
        got = ctx.render(sc, util.default_camera(0.0, 3), capi.make_params(L.KERNEL_GI, 160, 90, max_ray_depth=4, flags=pipe))
        assert_images_match(got, want, "synthetic GI, flags %d" % pipe, max_outliers=3)
    sc.release()


def test_full_size_properties(ctx):
    """1080p, BASELINE config 2 size: properties that need no oracle run."""
    sb, sc = gpu_scene(ctx, "cornell_box")
    w, h = 1920, 1080
    lin = ctx.render(sc, util.default_camera(), capi.make_params(L.KERNEL_BASIC_CU, w, h, kernel_mode=0))
    til = ctx.render(sc, util.default_camera(), capi.make_params(L.KERNEL_BASIC_CU, w, h, kernel_mode=1))
    util.assert_bit_equal(lin, til, "linear vs tile")  # tests/cuda_renderer_test.cc:117-180
    # a sub-window of the full-size image equals the oracle on those rows
    want = O.render(L.KERNEL_BASIC_CU, sb, util.default_camera(), w, h, rows=(500, 540), threads=0)
    util.assert_bit_equal(lin[500:540], want[500:540], "rows 500-540 at 1080p")
    # GI: 2 frames in one launch == 2 launches; band check against the oracle
    ctx.accum_reset()
    p2 = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
    two = ctx.render(sc, util.default_camera(0.0, 0), p2)
    acc = np.zeros((h, w, 3), np.float32)
    for f in range(2):
        O.accumulate(acc, O.render(L.KERNEL_GI, sb, util.default_camera(0.0, f), w, h, max_ray_depth=4,
                                   rows=(600, 620), threads=0), f)
    assert_images_match(two[600:620], acc[600:620], "GI rows 600-620 at 1080p", max_outliers=3)


@pytest.mark.parametrize("name", ["green_wall", "cornell_box", "cornell_box_lens", "single", "multi_leaf"])
def test_culling_is_output_identical(ctx, name):
    """LT_FLAG_CULL (opt-in) does less work than the reference traversal; on every test scene its output --
    hit ids, t/u/v, colours, GI samples -- is bit-identical to the exact mode."""
    sb, sc = gpu_scene(ctx, name)
    for yaw in (0.0, 0.04, -0.07):
        cam = util.default_camera(yaw, 2)
        a = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, 320, 200)
        b = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, 320, 200, flags=L.FLAG_CULL)
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1], b[1])
        util.assert_bit_equal(a[2], b[2], "t,u,v culled vs exact")
        for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_CUSTOM_BARY, L.KERNEL_ACCUMULATOR, L.KERNEL_GI):
            exact = ctx.render(sc, cam, capi.make_params(kernel, 200, 120, max_ray_depth=4))
            culled = ctx.render(sc, cam, capi.make_params(kernel, 200, 120, max_ray_depth=4, flags=L.FLAG_CULL))
            util.assert_bit_equal(culled, exact, "%s kernel %d culled vs exact" % (name, kernel))


def test_culling_on_a_synthetic_mesh(ctx, tmp_path):
    from lens_trace_b200 import host
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 160, 0x5EED)  # 51 212 triangles
    sb = host.load_scene_buffers(p)
    sc = ctx.upload(sb)
    cam = util.default_camera(0.0, 1)
    a = ctx.primary_hits(sc, cam, L.KERNEL_GI, 640, 360)
    b = ctx.primary_hits(sc, cam, L.KERNEL_GI, 640, 360, flags=L.FLAG_CULL)
    np.testing.assert_array_equal(a[0], b[0])
    util.assert_bit_equal(a[2], b[2])
    p_exact = capi.make_params(L.KERNEL_GI, 320, 180, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN,
                               flags=L.FLAG_STATS)
    p_cull = capi.make_params(L.KERNEL_GI, 320, 180, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN,
                              flags=L.FLAG_STATS | L.FLAG_CULL)
    ctx.accum_reset()
    exact = ctx.render(sc, cam, p_exact)
    n_exact = ctx.stats().node_tests
    ctx.accum_reset()
    culled = ctx.render(sc, cam, p_cull)
    n_cull = ctx.stats().node_tests
    util.assert_bit_equal(culled, exact, "synthetic GI culled vs exact")
    assert n_cull < n_exact  # it really does less work
    sc.release()


def test_bad_arguments_are_errors(ctx):
    sb, sc = gpu_scene(ctx, "cornell_box")
    with pytest.raises(capi.LtError):
        ctx.render(sc, util.default_camera(), capi.make_params(99, 10, 10))
    with pytest.raises(capi.LtError):
        ctx.render(sc, util.default_camera(), capi.make_params(L.KERNEL_BASIC_CU, 0, 10))
    bad = L.SceneBuffers(sb.nodes.copy(), sb.prims.copy(), sb.materials.copy(), sb.lights.copy())
    bad.nodes["offset"][0] = 10 ** 6
    with pytest.raises(capi.LtError):
        ctx.upload(bad)


def _model_prims(name_or_path):
    """Primitive records in Model (file) order, i.e. NOT yet ordered by any builder."""
    from lens_trace_b200 import host
    import os
    path = name_or_path if os.path.exists(name_or_path) else os.path.join(util.MODELS, name_or_path + ".obj")
    sb = host.load_scene_buffers(path)
    rng = np.random.default_rng(5)
    perm = rng.permutation(len(sb.prims))
    return sb.prims[perm].copy(), sb.materials.copy(), sb


@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "green_wall"])
def test_gpu_lbvh_builder(ctx, name):
    """lt_scene_build_lbvh: a valid tree in the reference layout (every primitive in exactly one leaf, boxes
    contain children, DFS order), traversed identically by the kernels and by the CPU oracle, and giving the
    same picture as the median-split tree."""
    from test_host import _check_tree
    prims, mats, median = _model_prims(name)
    sc = ctx.build_lbvh(prims, mats)
    sb, depth = ctx.download(sc)
    assert len(sb.nodes) == 2 * len(prims) - 1 and 1 <= depth <= 64
    _check_tree(sb)
    assert sorted(p.tobytes() for p in sb.prims) == sorted(p.tobytes() for p in prims)
    n = sb.lights["count"][0]
    assert n == median.lights["count"][0]
    for p in sb.lights["prims"][0][:n]:
        assert sb.materials["emission"][sb.prims["mat"][p]].max() > 0
    cam = util.default_camera(0.03, 1)
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, 200, 150)
    oids, ohit, otuv, _ = O.primary_hits(0, sb, cam, 200, 150)
    np.testing.assert_array_equal(hit, ohit)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv, "LBVH: kernels vs oracle on the same buffers")
    got = ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 160, 120, max_ray_depth=4))
    want = O.render(L.KERNEL_GI, sb, cam, 160, 120, max_ray_depth=4, threads=0)
    assert_images_match(got, want, "LBVH GI vs oracle", max_outliers=3)
    # same picture as the median-split tree for the deterministic kernel (ties at shared edges may pick the
    # other of two coplanar triangles, which has the same material here)
    _, msc = gpu_scene(ctx, name)
    a = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, 200, 150))
    b = ctx.render(msc, cam, capi.make_params(L.KERNEL_BASIC_CU, 200, 150))
    assert (np.abs(a - b).max(axis=-1) > 0).mean() < 0.002
    sc.release()


def test_gpu_lbvh_builder_large(ctx, tmp_path):
    from lens_trace_b200 import host
    from test_host import _check_tree
    p = str(tmp_path / "synth.obj")
    host.write_synthetic_scene(p, 200, 0x5EED)  # 80 012 triangles (exercises the parallel light selection)
    prims, mats, median = _model_prims(p)
    sc = ctx.build_lbvh(prims, mats)
    sb, depth = ctx.download(sc)
    _check_tree(sb)
    assert sb.lights["count"][0] == 2 and depth <= 64
    cam = util.default_camera()
    ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_GI, 320, 180)
    oids, ohit, otuv, _ = O.primary_hits(2, sb, cam, 320, 180)
    np.testing.assert_array_equal(ids, oids)
    util.assert_bit_equal(tuv, otuv)
    msc = ctx.upload(median)
    a = ctx.primary_hits(msc, cam, L.KERNEL_GI, 320, 180)
    assert (a[1] == hit).all()  # same hit mask as the median-split tree
    np.testing.assert_allclose(a[2][..., 0][hit == 1], tuv[..., 0][hit == 1], rtol=1e-5)
    msc.release()
    sc.release()


def test_depth_four_and_frame_stride(ctx):
    """imageDimensions[2] = 4 (three floats written per pixel, stride 4, basic.cu:344,361-363) and a frame stride
    (the frames one rank of a sample split renders) against the oracle."""
    sb, sc = gpu_scene(ctx, "cornell_box")
    w, h = 72, 40
    cam = util.default_camera(0.0, 1)
    got = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h, depth=4))
    want = O.render(L.KERNEL_BASIC_CU, sb, cam, w, h, depth=4)
    util.assert_bit_equal(got[..., :3], want[..., :3])
    for pipe in PIPES:
        ctx.accum_reset()
        p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, frames=3, frame_stride=4,
                             accum_mode=L.ACCUM_WEIGHTED_SUM, accum_weight=0.25, flags=pipe)
        got = ctx.render(sc, util.default_camera(0.0, 2), p)  # frameCount 2, 6, 10
        acc = np.zeros((h, w, 3), np.float32)
        for fc in (2, 6, 10):
            s = O.render(L.KERNEL_GI, sb, util.default_camera(0.0, fc), w, h, max_ray_depth=3, threads=0)
            acc = (acc + np.float32(0.25) * s).astype(np.float32)
        assert_images_match(got, acc, "weighted sum with stride", max_outliers=3)

"""Several camera views in one call (lt_render_views, lt_render_views_device, RenderExtensionB200::viewCount).  View v
of a call must equal, bit for bit, lt_accum_reset followed by lt_render of camera v alone with the same params, on every
kernel id, schedule flag and accumulation mode; the wavefront runs the views' (view, frame) pairs in one launch, the
megakernels one launch per view."""
import numpy as np
import pytest

import util
from lens_trace_b200 import capi, host, layouts as L

pytestmark = pytest.mark.gpu

KERNELS = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY, L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR,
           L.KERNEL_GI25, L.KERNEL_GI]
ACCUM = [(L.ACCUM_NONE, 0.0), (L.ACCUM_RUNNING_MEAN, 0.0), (L.ACCUM_WEIGHTED_SUM, 0.25)]


def cameras(n=3):
    """views with different positions, yaws and frameCounts (frameCount 0 discards an accumulator, > 0 folds into it)"""
    table = [(0.0, 2.5, -50.0, 0.0, 0), (1.5, 3.0, -45.0, 0.05, 3), (-2.0, 2.0, -55.0, -0.04, 7),
             (0.5, 2.7, -48.0, 0.02, 1), (-1.0, 2.4, -52.0, -0.01, 12)]
    return np.concatenate([L.make_camera(*table[k % len(table)][:4], frame_count=table[k % len(table)][4] + k // 5)
                           for k in range(n)])


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def scenes(ctx):
    up = {name: ctx.upload(util.scene(name)) for name in ("cornell_box", "cornell_box_lens")}
    yield up
    for sc in up.values():
        sc.release()


def singles(ctx, scene, cams, params):
    out = []
    for k in range(len(cams)):
        ctx.accum_reset()
        out.append(ctx.render(scene, cams[k:k + 1], params).copy())
    return out


def stats_of(ctx):
    s = ctx.stats()
    return np.array([s.rays, s.node_tests, s.tri_tests], np.uint64)


def check_views(ctx, scene, cams, params, what):
    got = ctx.render_views(scene, cams, params)
    want = singles(ctx, scene, cams, params)
    assert got.shape == (len(cams), params.height, params.width, params.depth)
    for v in range(len(cams)):
        util.assert_bit_equal(got[v], want[v], "%s, view %d" % (what, v))


@pytest.mark.parametrize("scene_name", ["cornell_box", "cornell_box_lens"])
@pytest.mark.parametrize("size", [(101, 75), (128, 96)])
@pytest.mark.parametrize("kernel", KERNELS)
def test_views_equal_single_renders(ctx, scenes, scene_name, size, kernel):
    w, h = size
    for frames in (1, 4):
        for mode, weight in ACCUM:
            p = capi.make_params(kernel, w, h, max_ray_depth=3, frames=frames, accum_mode=mode, accum_weight=weight)
            check_views(ctx, scenes[scene_name], cameras(), p, "kernel %d, %s, %dx%d, F=%d, accum %d"
                        % (kernel, scene_name, w, h, frames, mode))


SCHEDULES = [L.FLAG_WAVEFRONT, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT | L.FLAG_SERIAL, L.FLAG_CULL, L.FLAG_NO_THREADED,
             L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED]


@pytest.mark.parametrize("flags", SCHEDULES)
@pytest.mark.parametrize("kernel", [L.KERNEL_GI, L.KERNEL_ACCUMULATOR, L.KERNEL_GI25, L.KERNEL_BASIC_CU])
def test_views_under_every_schedule(ctx, scenes, flags, kernel):
    for frames in (1, 4):
        for mode, weight in ACCUM:
            p = capi.make_params(kernel, 101, 75, max_ray_depth=4, frames=frames, accum_mode=mode, accum_weight=weight,
                                 flags=flags)
            check_views(ctx, scenes["cornell_box"], cameras(), p, "flags %d, kernel %d, F=%d, accum %d"
                        % (flags, kernel, frames, mode))


def test_views_on_large_scene_paths():
    """device-built threaded copies, the tile-fetching k_flat_stream: the paths large scenes take"""
    with capi.Context(0) as c:
        c.debug_limits(0, 0)
        sc = c.upload(util.scene("cornell_box_lens"))
        for kernel in KERNELS:
            for flags in (0, L.FLAG_WAVEFRONT):
                for frames, (mode, weight) in ((1, ACCUM[0]), (3, ACCUM[1]), (2, ACCUM[2])):
                    p = capi.make_params(kernel, 101, 75, max_ray_depth=3, frames=frames, accum_mode=mode,
                                         accum_weight=weight, flags=flags)
                    check_views(c, sc, cameras(), p, "large-scene paths, kernel %d, flags %d, F=%d"
                                % (kernel, flags, frames))
        sc.release()


def test_batch_boundary_inside_a_view(ctx, scenes):
    """3 views x 3 frames on two streams: batches of 5 pairs, so the boundary falls inside view 1"""
    p = capi.make_params(L.KERNEL_GI, 128, 96, max_ray_depth=4, frames=3, accum_mode=L.ACCUM_RUNNING_MEAN,
                         flags=L.FLAG_WAVEFRONT)
    info = capi.plan_views(p, 3, 83, 8, 180 << 30, 148)
    assert info["pipeline"] == capi.PIPE_WAVEFRONT and info["batch_frames"] == 5 and info["streams"] == 2
    check_views(ctx, scenes["cornell_box"], cameras(), p, "batch boundary inside a view")
    p.flags |= L.FLAG_SERIAL
    check_views(ctx, scenes["cornell_box"], cameras(), p, "batch boundary inside a view, one stream")


def test_1080p_views_take_the_wavefront(ctx, scenes):
    """8 one-frame 1080p GI views hold enough paths for the wavefront: the planner picks it on its own"""
    p = capi.make_params(L.KERNEL_GI, 1920, 1080, max_ray_depth=4)
    sc = util.scene("cornell_box")
    single = capi.plan(p, len(sc.nodes), 8, 180 << 30, 148)
    views = capi.plan_views(p, 8, len(sc.nodes), 8, 180 << 30, 148)
    assert single["pipeline"] == capi.PIPE_PATH
    assert views["pipeline"] == capi.PIPE_WAVEFRONT
    check_views(ctx, scenes["cornell_box"], cameras(8), p, "1080p GI, 8 views")


@pytest.mark.parametrize("traced", [False, True])
@pytest.mark.parametrize("flags", [0, L.FLAG_WAVEFRONT, L.FLAG_MEGAKERNEL])
def test_views_stats_are_the_sum(ctx, scenes, traced, flags):
    flags |= L.FLAG_STATS | (L.FLAG_STATS_TRACED if traced else 0)
    for kernel in (L.KERNEL_GI, L.KERNEL_ACCUMULATOR, L.KERNEL_BASIC_CU):
        p = capi.make_params(kernel, 101, 75, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
        cams = cameras()
        got = ctx.render_views(scenes["cornell_box"], cams, p)
        total = stats_of(ctx)
        want = np.zeros(3, np.uint64)
        for k in range(len(cams)):
            ctx.accum_reset()
            single = ctx.render(scenes["cornell_box"], cams[k:k + 1], p)
            util.assert_bit_equal(got[k], single, "stats launch, view %d" % k)
            want += stats_of(ctx)
        assert total[0] > 0
        assert (total == want).all(), (kernel, flags, total, want)


def test_views_device_form(ctx, scenes):
    torch = pytest.importorskip("torch")
    cams = cameras()
    w, h = 101, 75
    for flags in (0, L.FLAG_WAVEFRONT):
        for mode, weight in ACCUM[1:]:
            p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=3, accum_mode=mode, accum_weight=weight,
                                 flags=flags)
            g = torch.Generator().manual_seed(5)
            start = torch.rand((len(cams), h, w, 3), generator=g, dtype=torch.float32)
            got = start.clone().cuda()
            ctx.render_views_device(scenes["cornell_box"], cams, p, got.data_ptr(), sync=True)
            for v in range(len(cams)):
                want = start[v].clone().cuda()
                ctx.render_device(scenes["cornell_box"], cams[v:v + 1], p, want.data_ptr(), sync=True)
                util.assert_bit_equal(got[v].cpu().numpy(), want.cpu().numpy(), "device form, flags %d, view %d"
                                      % (flags, v))
            # frameCount 0 discards the earlier accumulator (running mean), frameCount > 0 folds into it
            if mode == L.ACCUM_RUNNING_MEAN:
                fresh = ctx.render_views(scenes["cornell_box"], cams, p)
                assert (util.bits(got[0].cpu().numpy()) == util.bits(fresh[0])).all()
                assert (util.bits(got[1].cpu().numpy()) != util.bits(fresh[1])).any()


def test_views_leave_the_context_accumulator(ctx, scenes):
    p = capi.make_params(L.KERNEL_GI, 101, 75, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
    ctx.accum_reset()
    ctx.render(scenes["cornell_box"], util.default_camera(0.0, 0), p)
    before = np.empty((75, 101, 3), np.float32)
    ctx._check(ctx.lib.lt_accum_read(ctx.h, before.ctypes.data, before.size), "lt_accum_read")
    for flags in (0, L.FLAG_WAVEFRONT):
        p.flags = flags
        ctx.render_views(scenes["cornell_box"], cameras(), p)
    after = np.empty_like(before)
    ctx._check(ctx.lib.lt_accum_read(ctx.h, after.ctypes.data, after.size), "lt_accum_read")
    util.assert_bit_equal(after, before, "context accumulator after a views call")


def test_one_view_is_lt_render(ctx, scenes):
    cams = cameras(1)
    for flags in (0, L.FLAG_WAVEFRONT):
        p = capi.make_params(L.KERNEL_GI, 101, 75, max_ray_depth=4, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN,
                             flags=flags)
        check_views(ctx, scenes["cornell_box"], cams, p, "one view, flags %d" % flags)


def test_views_argument_errors(ctx, scenes):
    p = capi.make_params(L.KERNEL_GI, 32, 32)
    cams = cameras()
    lib = ctx.lib
    assert lib.lt_render_views(ctx.h, scenes["cornell_box"].h, cams.ctypes.data, 0, p, None) == capi.ERR_INVALID
    assert lib.lt_render_views(ctx.h, scenes["cornell_box"].h, None, 3, p, None) == capi.ERR_INVALID
    assert lib.lt_render_views_device(ctx.h, scenes["cornell_box"].h, cams.ctypes.data, -1, p, 1, 1) == capi.ERR_INVALID
    assert lib.lt_render_views_device(ctx.h, scenes["cornell_box"].h, cams.ctypes.data, 3, p, None, 1) == capi.ERR_INVALID


KERNEL_FILE = "examples/global_illumination/resources/kernels/global_illumination.cl"


def test_cpp_renderer_views():
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model)
    table = [(0.0, 2.5, -50.0, 0.0, 0), (1.5, 3.0, -45.0, 0.05, 3), (-2.0, 2.0, -55.0, -0.04, 7)]
    cams = []
    for x, y, z, yaw, fc in table:
        c = host.Camera(x, y, z, yaw)
        c.set_frame_count(fc)
        cams.append(c)
    w, h = 101, 75
    r = host.Renderer(host.PLATFORM_OPENCL)
    ext = host.make_extension(frames=3, accumulate=True, max_ray_depth=4, collect_stats=True, view_cameras=cams)
    got = r.render(KERNEL_FILE, w, h, accel, model, cams[0], ext=ext,
                   out=np.zeros((3, h, w, 3), np.float32))
    views_counts = (ext.rays, ext.nodeTests, ext.triTests)
    sums = np.zeros(3, np.uint64)
    for k, c in enumerate(cams):
        single = host.Renderer(host.PLATFORM_OPENCL)  # a fresh accumulator per view
        e1 = host.make_extension(frames=3, accumulate=True, max_ray_depth=4, collect_stats=True)
        want = single.render(KERNEL_FILE, w, h, accel, model, c, ext=e1)
        sums += np.array([e1.rays, e1.nodeTests, e1.triTests], np.uint64)
        util.assert_bit_equal(got[k], want, "RendererOpenCL, view %d" % k)
        single.close()
    assert tuple(int(x) for x in sums) == tuple(int(x) for x in views_counts)
    # a buffer below viewCount images is left untouched
    small = np.full((2, h, w, 3), 7.0, np.float32)
    r.render(KERNEL_FILE, w, h, accel, model, cams[0], ext=ext, out=small)
    assert (small == 7.0).all()
    r.close()
    for c in cams:
        c.close()
    accel.close()
    model.close()


def test_multi_gpu_views_equal_single_gpu():
    cams = cameras(5)
    p = capi.make_params(L.KERNEL_GI, 101, 75, max_ray_depth=4, frames=3, accum_mode=L.ACCUM_RUNNING_MEAN)
    with capi.Context(0) as one:
        sc = one.upload(util.scene("cornell_box"))
        want = one.render_views(sc, cams, p)
        sc.release()
    for n in util.group_sizes():
        p.split_mode = L.SPLIT_AUTO
        with util.device_group(n) as multi:
            sc = multi.upload(util.scene("cornell_box"))
            got = multi.render_views(sc, cams, p)
            p.split_mode = 1
            with pytest.raises(capi.LtError):
                multi.render_views(sc, cams, p)
            sc.release()
        util.assert_bit_equal(got, want, "multi-GPU views, %d devices" % n)

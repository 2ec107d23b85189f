"""lt_last_stats after a call: every field describes that call and reads 0 for what the call did not measure -- the
counters without LT_FLAG_STATS, the kernel time of an asynchronous call.  On a multi-GPU context, a device with no
share in a call adds nothing to the call's statistics, and a call refused for its parameters leaves the devices'
accumulators as they were.  The multi-GPU cases run on shared groups (util.device_group) on a machine with one GPU."""
import os

import numpy as np
import pytest

import util
from lens_trace_b200 import capi, host, layouts as L

pytestmark = pytest.mark.gpu

GI_FILE = "examples/global_illumination/resources/kernels/global_illumination.cl"


def rel_diff(a, b):
    return float((np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), 1e-3)).max())


def test_counters_of_a_call_without_stats():
    with capi.Context(0) as ctx:
        sc = ctx.upload(util.scene("cornell_box"))
        cam = util.default_camera()
        ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 96, 64, max_ray_depth=3, flags=L.FLAG_STATS))
        s = ctx.stats()
        assert s.rays > 0 and s.node_tests > 0 and s.tri_tests > 0
        ctx.render(sc, cam, capi.make_params(L.KERNEL_GI, 96, 64, max_ray_depth=3))
        s = ctx.stats()
        assert (s.rays, s.node_tests, s.tri_tests) == (0, 0, 0)
        assert s.kernel_ms > 0 and s.kernel_launches > 0
        sc.release()


def test_counters_through_the_renderer_extension():
    os.chdir(util.ROOT)  # resource paths are CWD-relative
    cam = host.Camera(0, 2.5, -50, 0)
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model)
    r = host.Renderer(host.PLATFORM_CUDA)
    counted = host.make_extension(frames=2, accumulate=True, max_ray_depth=3, collect_stats=True)
    r.render(GI_FILE, 96, 64, accel, model, cam, ext=counted)
    assert counted.rays > 0
    plain = host.make_extension(frames=2, accumulate=True, max_ray_depth=3, collect_stats=False)
    r.render(GI_FILE, 96, 64, accel, model, cam, ext=plain)
    assert (plain.rays, plain.nodeTests, plain.triTests) == (0, 0, 0)
    assert plain.kernelMilliseconds > 0
    r.close(); accel.close(); model.close(); cam.close()


def test_kernel_time_of_an_asynchronous_call():
    import torch
    w, h = 320, 200
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4)
    out = torch.empty((h, w, 3), dtype=torch.float32, device="cuda:0")
    with capi.Context(0) as ctx:
        sc = ctx.upload(util.scene("cornell_box"))
        cam = util.default_camera()
        ctx.render(sc, cam, p, want_output=False)
        synced = ctx.stats()
        assert synced.kernel_ms > 0 and synced.kernel_launches > 0
        ctx.render_device(sc, cam, p, out.data_ptr(), sync=False)
        s = ctx.stats()
        assert (s.kernel_ms, s.trace_ms, s.shade_ms, s.primary_shade_ms, s.accumulate_ms) == (0, 0, 0, 0, 0)
        assert s.kernel_launches == synced.kernel_launches
        torch.cuda.synchronize()
        sc.release()


def test_devices_without_a_share_add_nothing():
    for n in util.group_sizes():
        devices_without_a_share_add_nothing(n)


def devices_without_a_share_add_nothing(n):
    cam = util.default_camera()

    def samples(frames):
        return capi.make_params(L.KERNEL_GI, 64, 48, max_ray_depth=3, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                                split_mode=L.SPLIT_SAMPLES)

    def tiles(height):  # height 8 is one block of rows: device 0's alone
        return capi.make_params(L.KERNEL_GI, 64, height, max_ray_depth=3, split_mode=L.SPLIT_TILES)

    for params, busy in ((samples, 8), (tiles, 64)):
        idle = 1 if params is samples else 8
        with util.device_group(n) as many:
            sm = many.upload(util.scene("cornell_box"))
            many.render(sm, cam, params(idle), want_output=False)
            fresh = many.stats().kernel_launches
            many.render(sm, cam, params(busy), want_output=False)
            assert many.stats().kernel_launches > fresh
            many.render(sm, cam, params(idle), want_output=False)
            s = many.stats()
            assert s.kernel_launches == fresh, (params.__name__, s.kernel_launches, fresh)
            assert s.kernel_ms > 0
            sm.release()


@pytest.mark.parametrize("exchange", ["nccl", "p2p"])
def test_refused_call_leaves_the_accumulators(exchange, monkeypatch):
    """A (frames 0-3), the refused B (max_ray_depth 300), C (frames 4-7): C as after A alone."""
    util.skip_nccl_without_two_gpus(exchange)
    monkeypatch.setenv("LT_MULTI_EXCHANGE", exchange)
    for n in util.group_sizes():
        refused_call_leaves_the_accumulators(exchange, n)


def refused_call_leaves_the_accumulators(exchange, n):
    sb = util.scene("cornell_box")
    w, h = 160, 96

    def p(depth=4):
        return capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=depth, frames=4, accum_mode=L.ACCUM_RUNNING_MEAN,
                                split_mode=L.SPLIT_SAMPLES)

    with capi.Context(0) as one:
        s1 = one.upload(sb)
        one.render(s1, util.default_camera(0.0, 0), p(), want_output=False)
        want = one.render(s1, util.default_camera(0.0, 4), p())
        s1.release()
    got = []
    for refuse in (False, True):
        with util.device_group(n) as many:
            sm = many.upload(sb)
            many.render(sm, util.default_camera(0.0, 0), p(), want_output=False)
            if refuse:
                with pytest.raises(capi.LtError):
                    many.render(sm, util.default_camera(0.0, 4), p(depth=300))
            got.append(many.render(sm, util.default_camera(0.0, 4), p()))
            sm.release()
    if exchange == "p2p":
        util.assert_bit_equal(got[1], got[0], "C after a refused B vs C after A alone")
    for g in got:
        assert rel_diff(g, want) <= 1e-5, (exchange, rel_diff(g, want))

"""Destruction of contexts and scenes on the GPU: a context destroyed after work that fills every buffer, event pool and
stream it owns leaves nothing behind that changes the next context's results, and the stream a caller lent it
(lt_ctx_set_stream) outlives it.  Each run makes and destroys its own objects; later runs must reproduce the first bit
for bit."""
import os

import numpy as np
import pytest

import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu

GI_PLUGIN = os.path.join(util.ROOT, "tests", "plugins", "gi_plugin.cu")
W, H = 160, 120


def gi(w=W, h=H, **kw):
    return capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, **kw)


def dev(shape):
    import torch
    return torch.zeros(shape, dtype=torch.float32, device="cuda")


def test_the_callers_stream_outlives_the_context():
    import torch
    sb = util.scene("cornell_box")
    cam = util.default_camera(0.0, 0)
    p = gi(frames=4, accum_mode=L.ACCUM_RUNNING_MEAN)
    with capi.Context(0) as fresh:
        sc = fresh.upload(sb)
        want = dev((H, W, 3))
        fresh.render_device(sc, cam, p, want.data_ptr(), sync=True)
        sc.release()
    stream = torch.cuda.Stream()
    out = dev((H, W, 3))
    torch.cuda.synchronize()
    ctx = capi.Context(0)
    sc = ctx.upload(sb)
    ctx.set_stream(stream.cuda_stream)
    ctx.render_device(sc, cam, p, out.data_ptr(), sync=False)
    sc.release()
    ctx.close()  # synchronizes the caller's stream and leaves it alone
    with torch.cuda.stream(stream):
        copy = out * 1.0
    stream.synchronize()
    util.assert_bit_equal(out.cpu().numpy(), want.cpu().numpy(), "render on the caller's stream")
    util.assert_bit_equal(copy.cpu().numpy(), want.cpu().numpy(), "torch work on the stream after the context went")


def grown_context_run():
    """One context through every call that grows something it owns; returns its images and the scenes' byte counts."""
    import torch
    sb = util.scene("cornell_box")
    cam = util.default_camera(0.0, 0)
    images = {}
    with capi.Context(0) as ctx:
        sc = ctx.upload(sb)
        # timed wavefront call with statistics: the trace-event pool
        images["wavefront stats"] = ctx.render(sc, cam, gi(flags=L.FLAG_WAVEFRONT | L.FLAG_STATS))
        assert ctx.stats().trace_launches > 0
        # a pageable host image of more than 1 MB: the pinned stage, its events and the copier threads
        images["staged"] = ctx.render(sc, cam, gi(640, 480, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN))
        cams = np.stack([util.default_camera(y, 0) for y in (0.0, 0.1, 0.2)])
        images["views"] = ctx.render_views(sc, cams, gi(frames=2, accum_mode=L.ACCUM_RUNNING_MEAN,
                                                        flags=L.FLAG_WAVEFRONT))
        views = dev((3, H, W, 3))
        ctx.render_views_device(sc, cams, gi(frames=2, accum_mode=L.ACCUM_RUNNING_MEAN), views.data_ptr(), sync=True)
        images["views device"] = views.cpu().numpy()
        out, m2 = dev((H, W, 3)), dev((H, W, 3))
        mask = torch.from_numpy(np.random.default_rng(7).random((H, W)) < 0.4).to(torch.uint8).cuda()
        ctx.render_masked_device(sc, cam, gi(frames=3, accum_mode=L.ACCUM_RUNNING_MEAN), out.data_ptr(),
                                 mask.data_ptr(), m2.data_ptr(), sync=True)
        images["masked"], images["masked m2"] = out.cpu().numpy(), m2.cpu().numpy()
        adaptive = gi(frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
        mean, frames, _ = ctx.render_adaptive(sc, cam, adaptive, 0.1, round_frames=2, max_frames=8)
        images["adaptive"], images["adaptive frames"] = mean, frames.view(np.float32)
        out, m2 = dev((H, W, 3)), dev((H, W, 3))
        counts = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        ctx.render_adaptive_device(sc, cam, adaptive, out.data_ptr(), m2.data_ptr(), counts.data_ptr(),
                                   target=0.1, round_frames=2, max_frames=8, sync=True)
        images["adaptive device"], images["adaptive device m2"] = out.cpu().numpy(), m2.cpu().numpy()
        pid = ctx.plugin_load(GI_PLUGIN)
        p = capi.make_params(0, W, H, frames=3, accum_mode=L.ACCUM_RUNNING_MEAN)
        p.block_x, p.block_y = 8, 8
        ctx.accum_reset()
        images["plug-in frames"] = ctx.render_plugin_frames(sc, cam, pid, p)
        ids, hit, tuv = ctx.primary_hits(sc, cam, L.KERNEL_BASIC_CU, W, H)
        images["primary hits"] = np.concatenate([ids.view(np.float32).ravel(), hit.view(np.float32).ravel(),
                                                 tuv.ravel()])
        ctx.refit(sc, sb.prims)
        images["refitted"] = ctx.render(sc, cam, gi())
        # device-built threaded copies
        ctx.debug_limits(threaded_max_nodes=0, stream_min_nodes=100000)
        big = ctx.upload(sb)
        images["device-built copies"] = ctx.render(big, cam, capi.make_params(L.KERNEL_BASIC_CU, W, H))
        scene_bytes = (ctx.scene_bytes(sc), ctx.scene_bytes(big))
        big.release()
        sc.release()
    return images, scene_bytes


def test_a_fully_grown_context_tears_down_cleanly():
    first, first_bytes = grown_context_run()
    assert all(b > 0 for b in first_bytes)
    for run in (2, 3):
        images, scene_bytes = grown_context_run()
        assert scene_bytes == first_bytes, run
        assert images.keys() == first.keys()
        for what in first:
            util.assert_bit_equal(images[what], first[what], "run %d, %s" % (run, what))


def test_a_shared_group_tears_down_cleanly(monkeypatch):
    monkeypatch.setenv("LT_MULTI_EXCHANGE", "p2p")
    sb = util.scene("cornell_box")
    cam = util.default_camera(0.0, 0)
    p = gi(frames=6, accum_mode=L.ACCUM_RUNNING_MEAN, split_mode=L.SPLIT_SAMPLES)
    runs = []
    for _ in range(3):
        with capi.Context.shared(0, 3) as group:
            sc = group.upload(sb)
            runs.append(group.render(sc, cam, p))  # the exchange buffers and the members' events
            sc.release()
    for run in (1, 2):
        util.assert_bit_equal(runs[run], runs[0], "run %d" % (run + 1))

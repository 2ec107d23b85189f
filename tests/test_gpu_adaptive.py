"""Adaptive sampling in the library (lt_render_adaptive, lt_render_adaptive_device): the result equals the torch loop of
INTEGRATION section 5d built on lt_render_masked_device, bit for bit (mean, m2 and frame counts), every pixel equals a
plain render of its own frame count, and the host form, the row partition of several devices and the C++ renderer give
the same pixels."""
import ctypes as C
import os

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, host, layouts as L

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STOCHASTIC = [L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR, L.KERNEL_GI25, L.KERNEL_GI]
DETERMINISTIC = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY]
W, H = 101, 75
NAN = np.uint32(0x7fc0beef)


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


def cam(frame_count):
    return util.default_camera(0.03, frame_count)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host_of(t):
    return t.cpu().numpy()


def f32(x):
    return torch.tensor(x, dtype=torch.float32, device="cuda")


def params(kernel, w, h, frames, flags=0):
    return capi.make_params(kernel, w, h, max_ray_depth=4, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)


def schedule(frames, round_frames, max_frames):
    r = [frames]
    while sum(r) < max_frames:
        r.append(min(round_frames or frames, max_frames - sum(r)))
    return r


def loop_5d(ctx, sc, kernel, w, h, c, start, start_m2, target, frames, round_frames, max_frames, floor=1e-4, flags=0):
    """the loop of INTEGRATION section 5d, with its rule restated in torch float32 ops: returns mean, m2, frame counts,
    rounds, pixel-frames, unconverged pixels and the summed stats counters / launches of the masked calls"""
    out, m2 = dev(start), dev(start_m2)
    n = torch.full((h, w), 0, dtype=torch.int32, device="cuda")
    active = torch.ones((h, w), dtype=torch.bool, device="cuda")
    mask = None
    done, rounds, pixel_frames, f = 0, 0, 0, frames
    counters = np.zeros(3, np.uint64)
    launches = 0
    while True:
        p = params(kernel, w, h, f, flags)
        ctx.render_masked_device(sc, cam(c + done), p, out.data_ptr(), mask.data_ptr() if mask is not None else None,
                                 m2.data_ptr(), sync=True)
        s = ctx.stats()
        counters += np.array([s.rays, s.node_tests, s.tri_tests], np.uint64)
        launches += s.kernel_launches
        rounds += 1
        pixel_frames += int(active.sum()) * f
        done += f
        nn = c + done
        n[active] = nn
        d = f32(float(nn)) * f32(float(nn - 1))
        err = (torch.sqrt(m2 / d) / out[..., :3].clamp_min(f32(floor))).amax(dim=2)
        go = (err > f32(target)) & active
        if done == max_frames:
            unconverged = int(go.sum())
            break
        if not bool(go.any()):
            unconverged = 0
            break
        f = min(round_frames or frames, max_frames - done)
        active = go
        mask = go.to(torch.uint8).contiguous()
    torch.cuda.synchronize()
    return dict(out=host_of(out), m2=host_of(m2), n=host_of(n).astype(np.uint32), rounds=rounds,
                pixel_frames=pixel_frames, unconverged=unconverged, counters=counters, launches=launches)


def adaptive_device(ctx, sc, kernel, w, h, c, start, start_m2, target, frames, round_frames, max_frames, floor=0.0,
                    flags=0, frames_start=None):
    out, m2 = dev(start), dev(start_m2)
    fr = dev(np.full((h, w), 0xDEADBEEF, np.uint32).view(np.int32) if frames_start is None else frames_start)
    res = ctx.render_adaptive_device(sc, cam(c), params(kernel, w, h, frames, flags), out.data_ptr(), m2.data_ptr(),
                                     fr.data_ptr(), target=target, round_frames=round_frames, max_frames=max_frames,
                                     floor=floor, sync=True)
    return dict(out=host_of(out), m2=host_of(m2), n=host_of(fr).view(np.uint32), rounds=res.rounds,
                pixel_frames=res.pixel_frames, unconverged=res.pixels_unconverged, stats=ctx.stats())


def assert_same(got, want, what):
    util.assert_bit_equal(got["out"], want["out"], what + ", mean")
    util.assert_bit_equal(got["m2"], want["m2"], what + ", m2")
    util.assert_bit_equal(got["n"], want["n"], what + ", frame counts")
    assert (got["rounds"], got["pixel_frames"], got["unconverged"]) == \
        (want["rounds"], want["pixel_frames"], want["unconverged"]), what


def zeros(w=W, h=H):
    return np.zeros((h, w, 3), np.float32)


@pytest.mark.parametrize("flags", [L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT])
@pytest.mark.parametrize("scene_name", ["cornell_box", "cornell_box_lens"])
@pytest.mark.parametrize("kernel", STOCHASTIC)
def test_equals_the_5d_loop(ctx, scenes, kernel, scene_name, flags):
    sc = scenes[scene_name]
    for target, frames, rf, mx in ((0.1, 4, 4, 16), (0.05, 2, 3, 14)):
        want = loop_5d(ctx, sc, kernel, W, H, 0, zeros(), zeros(), target, frames, rf, mx, flags=flags)
        got = adaptive_device(ctx, sc, kernel, W, H, 0, zeros(), zeros(), target, frames, rf, mx, flags=flags)
        assert_same(got, want, "kernel %d, %s, flags %d, target %g" % (kernel, scene_name, flags, target))
        if kernel in (L.KERNEL_GI25, L.KERNEL_GI):
            assert want["rounds"] >= 2, "the case should take more than one round"


def test_equals_the_5d_loop_at_1080p(ctx, scenes):
    """the section 5d parameters (16 + 3 x 16 frames, 5 %) at 1080p on the default plan: the wavefront on full and
    partial lists"""
    w, h = 1920, 1080
    z = zeros(w, h)
    want = loop_5d(ctx, scenes["cornell_box"], L.KERNEL_GI, w, h, 0, z, z, 0.05, 16, 16, 64)
    got = adaptive_device(ctx, scenes["cornell_box"], L.KERNEL_GI, w, h, 0, z, z, 0.05, 16, 16, 64)
    assert_same(got, want, "1080p GI")
    assert want["rounds"] >= 2 and 0 < want["pixel_frames"] < 64 * w * h


def test_continuation_from_held_frames(ctx, scenes):
    """the device form from c = 5 frames already in out and m2"""
    sc = scenes["cornell_box"]
    out, m2 = dev(zeros()), dev(zeros())
    ctx.render_masked_device(sc, cam(0), params(L.KERNEL_GI, W, H, 5), out.data_ptr(), None, m2.data_ptr(), sync=True)
    start, start_m2 = host_of(out), host_of(m2)
    for frames in (1, 3):
        want = loop_5d(ctx, sc, L.KERNEL_GI, W, H, 5, start, start_m2, 0.08, frames, 2, 11)
        got = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 5, start, start_m2, 0.08, frames, 2, 11)
        assert_same(got, want, "continuation, %d frames first" % frames)


def test_each_pixel_is_a_plain_render_of_its_frames(ctx, scenes):
    sc = scenes["cornell_box_lens"]
    got = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 4, 4, 20)
    counts = np.unique(got["n"])
    assert len(counts) >= 2, counts
    for n in counts:
        plain = dev(zeros())
        ctx.render_device(sc, cam(0), params(L.KERNEL_GI, W, H, int(n)), plain.data_ptr(), sync=True)
        sel = got["n"] == n
        util.assert_bit_equal(got["out"][sel], host_of(plain)[sel], "pixels of %d frames" % n)


def test_running_mean_against_the_oracle(ctx, scenes):
    """small image: every pixel's mean equals oracle.accumulate over its own number of the oracle's frames"""
    sb = util.scene("cornell_box")
    w, h = 48, 36
    sc = scenes["cornell_box"]
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
    mean, n, res = ctx.render_adaptive(sc, cam(0), p, 0.1, round_frames=2, max_frames=6)
    assert res.rounds >= 2
    acc = np.zeros((h, w, 3), np.float32)
    for k in range(6):
        O.accumulate(acc, O.render(L.KERNEL_GI, sb, cam(k), w, h, max_ray_depth=3), k)
        sel = n == k + 1
        util.assert_bit_equal(mean[sel], acc[sel], "pixels of %d frames against the oracle" % (k + 1))
    assert set(np.unique(n)) <= {2, 4, 6}


def test_host_form_equals_the_device_form(ctx, scenes):
    sc = scenes["cornell_box"]
    for c, frames in ((0, 4), (3, 2)):
        want = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, c, zeros(), zeros(), 0.1, frames, 3, 16)
        mean, n, res = ctx.render_adaptive(sc, cam(c), params(L.KERNEL_GI, W, H, frames), 0.1, round_frames=3,
                                           max_frames=16)
        util.assert_bit_equal(mean, want["out"], "host form, c = %d" % c)
        util.assert_bit_equal(n, want["n"], "host form frame counts, c = %d" % c)
        assert (res.rounds, res.pixel_frames, res.pixels_unconverged) == \
            (want["rounds"], want["pixel_frames"], want["unconverged"])
    # depth 4: the mean has a fourth float per pixel that nothing writes
    p4 = capi.make_params(L.KERNEL_GI, W, H, depth=4, max_ray_depth=4, frames=4, accum_mode=L.ACCUM_RUNNING_MEAN)
    mean4, n4, _ = ctx.render_adaptive(sc, cam(0), p4, 0.1, round_frames=3, max_frames=16)
    want = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 4, 3, 16)
    util.assert_bit_equal(mean4[..., :3], want["out"], "depth 4")
    util.assert_bit_equal(n4, want["n"], "depth 4 frame counts")


def accum_read(ctx, floats):
    a = np.zeros(floats, np.float32)
    ctx._check(ctx.lib.lt_accum_read(ctx.h, a.ctypes.data, a.size), "lt_accum_read")
    return a


def test_context_accumulator_is_left_alone(ctx, scenes):
    sc = scenes["cornell_box"]
    p = params(L.KERNEL_GI, W, H, 3)
    ctx.accum_reset()
    ctx.render(sc, cam(0), p)
    before = accum_read(ctx, W * H * 3)
    ctx.render_adaptive(sc, cam(0), params(L.KERNEL_GI, W, H, 4), 0.1)
    util.assert_bit_equal(accum_read(ctx, W * H * 3), before, "context accumulator")


def test_tiny_target_runs_every_pixel_to_max_frames(ctx, scenes):
    sc = scenes["cornell_box"]
    want = loop_5d(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 1e-9, 4, 5, 17)
    got = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 1e-9, 4, 5, 17)
    assert_same(got, want, "tiny target")
    assert got["rounds"] == len(schedule(4, 5, 17)) == 4  # 4, 5, 5, then a shorter 3
    assert got["unconverged"] > 0 and got["unconverged"] == want["unconverged"]


def test_huge_target_is_one_masked_call(ctx, scenes):
    sc = scenes["cornell_box"]
    out, m2 = dev(zeros()), dev(zeros())
    ctx.render_masked_device(sc, cam(0), params(L.KERNEL_GI, W, H, 4), out.data_ptr(), None, m2.data_ptr(), sync=True)
    got = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 1e30, 4, 4, 16)
    util.assert_bit_equal(got["out"], host_of(out), "mean")
    util.assert_bit_equal(got["m2"], host_of(m2), "m2")
    assert (got["n"] == 4).all()
    assert (got["rounds"], got["pixel_frames"], got["unconverged"]) == (1, 4 * W * H, 0)


@pytest.mark.parametrize("kernel", DETERMINISTIC)
def test_deterministic_kernels_stop_after_one_round(ctx, scenes, kernel):
    for scene_name in ("cornell_box", "cornell_box_lens"):
        sc = scenes[scene_name]
        got = adaptive_device(ctx, sc, kernel, W, H, 0, zeros(), zeros(), 1e-9, 2, 2, 10)
        plain = dev(zeros())
        ctx.render_device(sc, cam(0), params(kernel, W, H, 2), plain.data_ptr(), sync=True)
        util.assert_bit_equal(got["out"], host_of(plain), "kernel %d, %s" % (kernel, scene_name))
        assert (got["m2"] == 0).all() and got["rounds"] == 1 and got["unconverged"] == 0


@pytest.mark.parametrize("flags", [0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_STATS])
def test_list_order_does_not_matter(ctx, scenes, flags):
    sc = scenes["cornell_box"]
    a = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12, flags=flags)
    ctx.debug_list_order(True)
    try:
        b = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12, flags=flags)
    finally:
        ctx.debug_list_order(False)
    assert_same(b, a, "reversed lists, flags %d" % flags)
    assert b["stats"].kernel_launches == a["stats"].kernel_launches + a["rounds"]  # one reversal per list


def test_large_scene_paths():
    """device-built threaded copies and the large-scene schedule (limits lowered), against the 5d loop"""
    with capi.Context(0) as c:
        c.debug_limits(0, 0)
        sc = c.upload(util.scene("cornell_box_lens"))
        for kernel in (L.KERNEL_LIGHTING25, L.KERNEL_GI, L.KERNEL_BASIC_CU):
            for flags in (0, L.FLAG_WAVEFRONT):
                if kernel == L.KERNEL_BASIC_CU and flags:
                    continue
                want = loop_5d(c, sc, kernel, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12, flags=flags)
                got = adaptive_device(c, sc, kernel, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12, flags=flags)
                assert_same(got, want, "large-scene paths, kernel %d, flags %d" % (kernel, flags))
        sc.release()


@pytest.mark.parametrize("flags", [L.FLAG_STATS, L.FLAG_STATS | L.FLAG_STATS_TRACED])
def test_stats_are_the_sum_of_the_masked_calls(ctx, scenes, flags):
    sc = scenes["cornell_box"]
    want = loop_5d(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12, flags=flags)
    got = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12, flags=flags)
    assert_same(got, want, "stats, flags %d" % flags)
    s = got["stats"]
    assert (s.rays, s.node_tests, s.tri_tests) == tuple(int(x) for x in want["counters"])
    assert s.rays > 0
    # each masked call compacts its own mask; the adaptive call compacts once and selects after every round
    assert s.kernel_launches == want["launches"] + 1


@pytest.mark.parametrize("parts", [2, 3, 8])
def test_row_parts_assemble_the_one_part_call(ctx, scenes, parts):
    """lt_debug_ctx_adaptive_part: the rows each device of a `parts`-device context renders, on one GPU; both forms"""
    sc = scenes["cornell_box_lens"]
    p = params(L.KERNEL_GI, W, H, 3)
    whole = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, zeros(), zeros(), 0.1, 3, 3, 12)
    nan = np.full((H, W, 3), NAN, np.uint32).view(np.float32)
    nan_frames = np.full((H, W), 0xDEADBEEF, np.uint32)
    out_dev = np.full((H, W, 3), NAN, np.uint32).view(np.float32)
    n_dev = nan_frames.copy()
    out_host = nan.copy()
    n_host = nan_frames.copy()
    pixel_frames = 0
    try:
        for g in range(parts):
            ctx.debug_adaptive_part(parts, g)
            got = adaptive_device(ctx, sc, L.KERNEL_GI, W, H, 0, nan, nan, 0.1, 3, 3, 12,
                                  frames_start=nan_frames.view(np.int32))
            mine = np.zeros(H, bool)
            mine[capi.tile_rows(H, parts, g)] = True
            util.assert_bit_equal(got["out"][~mine], nan[~mine], "rows of other parts, mean")
            util.assert_bit_equal(got["m2"][~mine], nan[~mine], "rows of other parts, m2")
            util.assert_bit_equal(got["n"][~mine], nan_frames[~mine], "rows of other parts, frames")
            out_dev[mine], n_dev[mine] = got["out"][mine], got["n"][mine]
            pixel_frames += got["pixel_frames"]
            # the host form writes its own rows only
            a = capi.make_adaptive(0.1, 12, 3)
            res = capi.AdaptiveResult()
            ctx._check(ctx.lib.lt_render_adaptive(ctx.h, sc.h, cam(0).ctypes.data, C.byref(p), C.byref(a),
                                                  out_host.ctypes.data, n_host.ctypes.data, C.byref(res)),
                       "lt_render_adaptive")
    finally:
        ctx.debug_adaptive_part(1, 0)
    util.assert_bit_equal(out_dev, whole["out"], "device form, %d parts assembled" % parts)
    util.assert_bit_equal(n_dev, whole["n"], "device form frame counts, %d parts assembled" % parts)
    util.assert_bit_equal(out_host, whole["out"], "host form, %d parts assembled" % parts)
    util.assert_bit_equal(n_host, whole["n"], "host form frame counts, %d parts assembled" % parts)
    assert pixel_frames == whole["pixel_frames"]


def test_argument_errors_leave_the_outputs(ctx, scenes):
    sc = scenes["cornell_box"]
    lib = ctx.lib
    start = np.full((H, W, 3), NAN, np.uint32).view(np.float32)
    out, m2 = dev(start), dev(start)
    res = capi.AdaptiveResult()
    cams = cam(0)

    def call(p, a, o=out.data_ptr(), m=m2.data_ptr(), f=None):
        return lib.lt_render_adaptive_device(ctx.h, sc.h, cams.ctypes.data, C.byref(p), C.byref(a), C.c_void_p(o),
                                             C.c_void_p(m) if m else None, C.c_void_p(f) if f else None, C.byref(res), 1)

    good_p, good_a = params(L.KERNEL_GI, W, H, 4), capi.make_adaptive(0.1, 16)
    assert call(capi.make_params(L.KERNEL_GI, W, H, frames=4), good_a) == capi.ERR_INVALID
    assert call(good_p, capi.make_adaptive(0.0, 16)) == capi.ERR_INVALID
    assert call(good_p, good_a, m=None) == capi.ERR_INVALID
    assert "device_out and device_m2 are required" in lib.lt_last_error(ctx.h).decode()
    host_buf = np.zeros((H, W, 3), np.float32)
    assert call(good_p, good_a, o=host_buf.ctypes.data) == capi.ERR_INVALID
    assert "device_out is not device memory" in lib.lt_last_error(ctx.h).decode()
    assert call(good_p, good_a, m=m2.data_ptr() + 2) == capi.ERR_INVALID
    assert "device_m2 is not 4-byte aligned" in lib.lt_last_error(ctx.h).decode()
    assert call(good_p, good_a, f=out.data_ptr() + 1) == capi.ERR_INVALID
    assert "device_frames is not 4-byte aligned" in lib.lt_last_error(ctx.h).decode()
    torch.cuda.synchronize()
    util.assert_bit_equal(host_of(out), start, "out after the errors")
    util.assert_bit_equal(host_of(m2), start, "m2 after the errors")


KERNEL_FILE = "examples/global_illumination/resources/kernels/global_illumination.cl"


def test_cpp_renderers_equal_the_host_form():
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model)
    w, h = 101, 75
    with capi.Context(0) as c:
        sc = c.upload(accel.buffers())
        want, want_n, res = c.render_adaptive(sc, L.make_camera(0, 2.5, -50, 0.0, 0), params(L.KERNEL_GI, w, h, 4),
                                              0.1, round_frames=2, max_frames=12)
        sc.release()
    assert res.rounds >= 2
    camera = host.Camera(0, 2.5, -50, 0.0)
    for platform in (host.PLATFORM_CUDA, host.PLATFORM_OPENCL):
        r = host.Renderer(platform)
        n = np.zeros((h, w), np.uint32)
        ext = host.make_extension(frames=4, accumulate=True, max_ray_depth=4, adaptive_error=0.1,
                                  adaptive_round_frames=2, adaptive_max_frames=12, pixel_frames=n)
        got = r.render(KERNEL_FILE, w, h, accel, model, camera, ext=ext)
        util.assert_bit_equal(got, want, "platform %d" % platform)
        util.assert_bit_equal(n, want_n, "platform %d, pixel frames" % platform)
        assert ext.adaptiveRounds == res.rounds and ext.kernelMilliseconds > 0
        # adaptiveMaxFrames 0: frames + 3 rounds
        ext = host.make_extension(frames=4, accumulate=True, max_ray_depth=4, adaptive_error=1e-9)
        r.render(KERNEL_FILE, w, h, accel, model, camera, ext=ext)
        assert ext.adaptiveRounds == 4
        # refused combinations leave the buffer untouched
        seeded = np.full((h, w, 3), NAN, np.uint32).view(np.float32)
        refused = [host.make_extension(frames=4, accumulate=False, adaptive_error=0.1),
                   host.make_extension(frames=4, accumulate=True, adaptive_error=0.1, split=1),
                   host.make_extension(frames=4, accumulate=True, adaptive_error=0.1, view_cameras=[camera, camera])]
        for e in refused:
            buf = seeded.copy() if e.viewCount < 2 else np.full((2, h, w, 3), NAN, np.uint32).view(np.float32)
            r.render(KERNEL_FILE, w, h, accel, model, camera, ext=e, out=buf)
            assert (buf.view(np.uint32) == NAN).all()
        plug = os.path.join(util.ROOT, "tests", "plugins", "gi_plugin.cu")
        buf = seeded.copy()
        r.render(plug, w, h, accel, model, camera, ext=host.make_extension(frames=4, accumulate=True, adaptive_error=0.1),
                 out=buf)
        assert (buf.view(np.uint32) == NAN).all()
        r.close()
    camera.close()
    accel.close()
    model.close()


def test_multi_gpu_equals_one_gpu():
    sb = util.scene("cornell_box_lens")
    w, h = 320, 203
    p = params(L.KERNEL_GI, w, h, 4)
    with capi.Context(0) as one:
        sc = one.upload(sb)
        want, want_n, want_res = one.render_adaptive(sc, cam(0), p, 0.08, round_frames=4, max_frames=16)
        sc.release()
    sizes = sorted({2, min(torch.cuda.device_count(), 8)}) if torch.cuda.device_count() >= 2 else util.group_sizes()
    for G in sizes:
        with util.device_group(G) as multi:
            sc = multi.upload(sb)
            for split in (L.SPLIT_AUTO, L.SPLIT_TILES):
                p.split_mode = split
                got, got_n, res = multi.render_adaptive(sc, cam(0), p, 0.08, round_frames=4, max_frames=16)
                util.assert_bit_equal(got, want, "%d GPUs, split %d" % (G, split))
                util.assert_bit_equal(got_n, want_n, "%d GPUs, split %d, frames" % (G, split))
                assert (res.pixel_frames, res.pixels_unconverged) == (want_res.pixel_frames, want_res.pixels_unconverged)
            p.split_mode = L.SPLIT_SAMPLES
            with pytest.raises(capi.LtError):
                multi.render_adaptive(sc, cam(0), p, 0.08, round_frames=4, max_frames=16)
            p.split_mode = L.SPLIT_AUTO
            sc.release()

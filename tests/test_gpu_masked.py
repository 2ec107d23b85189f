"""Masked continuation of accumulated renders (lt_render_masked_device): every masked pixel gets exactly what
lt_render_device gives it, bit for bit, pixels outside the mask keep their bytes, and m2 holds the Welford sums of the
frame samples beside the running mean.  Torch allocates the device buffers."""
import ctypes as C

import numpy as np
import pytest

import lt_oracle as O
import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

KERNELS = [L.KERNEL_BASIC_CU, L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY, L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR,
           L.KERNEL_GI25, L.KERNEL_GI]
STOCHASTIC = [L.KERNEL_LIGHTING25, L.KERNEL_ACCUMULATOR, L.KERNEL_GI25, L.KERNEL_GI]
W, H = 101, 75
NAN = np.uint32(0x7fc0beef)  # a quiet NaN with a payload: bytes outside the mask must keep it


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


def host(t):
    return t.cpu().numpy()


def plain(ctx, scene, params, start, frame_count):
    """lt_render_device from `start` (host array): the result every masked pixel must have"""
    out = dev(start)
    ctx.render_device(scene, cam(frame_count), params, out.data_ptr(), sync=True)
    return host(out)


def masked(ctx, scene, params, start, frame_count, mask=None, m2=None):
    out = dev(start)
    m = dev(mask.astype(np.uint8)) if mask is not None else None
    t2 = dev(m2) if m2 is not None else None
    ctx.render_masked_device(scene, cam(frame_count), params, out.data_ptr(), m.data_ptr() if m is not None else None,
                             t2.data_ptr() if t2 is not None else None, sync=True)
    return host(out), (host(t2) if t2 is not None else None)


def nan_outside(a, mask):
    """a copy of `a` whose floats of the pixels outside `mask` hold the NaN pattern"""
    b = np.array(a, np.float32, copy=True)
    b.view(np.uint32)[~mask] = NAN
    return b


def random_mask(seed, fraction=0.3, shape=(H, W)):
    return np.random.default_rng(seed).random(shape) < fraction


def assert_masked(got, want_in, want_out, mask, what):
    util.assert_bit_equal(got[mask], want_in[mask], what + ", masked pixels")
    util.assert_bit_equal(got[~mask], want_out[~mask], what + ", pixels outside the mask")


@pytest.mark.parametrize("scene_name", ["cornell_box", "cornell_box_lens"])
@pytest.mark.parametrize("flags", [0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_NO_THREADED])
@pytest.mark.parametrize("kernel", KERNELS)
def test_full_and_null_mask_equal_lt_render_device(ctx, scenes, scene_name, flags, kernel):
    sc = scenes[scene_name]
    start = np.random.default_rng(kernel).random((H, W, 3), dtype=np.float32)
    full = np.ones((H, W), bool)
    for frames, fc, (mode, weight) in ((1, 0, (L.ACCUM_NONE, 0.0)), (3, 2, (L.ACCUM_RUNNING_MEAN, 0.0)),
                                       (2, 5, (L.ACCUM_WEIGHTED_SUM, 0.25))):
        p = capi.make_params(kernel, W, H, max_ray_depth=3, frames=frames, accum_mode=mode, accum_weight=weight,
                             flags=flags)
        want = plain(ctx, sc, p, start, fc)
        what = "kernel %d, %s, flags %d, accum %d" % (kernel, scene_name, flags, mode)
        util.assert_bit_equal(masked(ctx, sc, p, start, fc, full)[0], want, what + ", full mask")
        util.assert_bit_equal(masked(ctx, sc, p, start, fc)[0], want, what + ", NULL mask")


def continuation(ctx, sc, kernel, flags, seed):
    """4 frames on every pixel (with m2), then 5 more from frameCount 4 under a random mask; outside the mask out and m2
    hold the NaN pattern before the second call"""
    first = capi.make_params(kernel, W, H, max_ray_depth=3, frames=4, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
    zero = np.zeros((H, W, 3), np.float32)
    out4, m2_4 = masked(ctx, sc, first, zero, 0, None, zero)
    ref9 = capi.make_params(kernel, W, H, max_ray_depth=3, frames=9, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
    out9, m2_9 = masked(ctx, sc, ref9, zero, 0, None, zero)
    util.assert_bit_equal(out4, plain(ctx, sc, first, zero, 0), "4 frames with m2 against lt_render_device")
    util.assert_bit_equal(out9, plain(ctx, sc, ref9, zero, 0), "9 frames with m2 against lt_render_device")
    mask = random_mask(seed)
    more = capi.make_params(kernel, W, H, max_ray_depth=3, frames=5, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
    got, got2 = masked(ctx, sc, more, nan_outside(out4, mask), 4, mask, nan_outside(m2_4, mask))
    what = "kernel %d, flags %d" % (kernel, flags)
    assert_masked(got, out9, nan_outside(out4, mask), mask, what)
    assert_masked(got2, m2_9, nan_outside(m2_4, mask), mask, what + ", m2")
    # and without m2
    got, _ = masked(ctx, sc, more, nan_outside(out4, mask), 4, mask)
    assert_masked(got, out9, nan_outside(out4, mask), mask, what + ", no m2")


SCHEDULES = [0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_SERIAL, L.FLAG_CULL, L.FLAG_STATS,
             L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED]


@pytest.mark.parametrize("flags", SCHEDULES)
@pytest.mark.parametrize("kernel", KERNELS)
def test_continuation_under_a_random_mask(ctx, scenes, kernel, flags):
    """the wavefront runs the 5 frames in batches of 3 on two streams: a batch boundary inside the call, overlapped"""
    if flags & L.FLAG_WAVEFRONT and flags & L.FLAG_SERIAL == 0:
        info = capi.plan_masked(capi.make_params(kernel, W, H, max_ray_depth=3, frames=5,
                                                 accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags), 2000, 83, 8, 180 << 30, 148)
        if kernel in STOCHASTIC:
            assert info["batch_frames"] == 3 and info["streams"] == 2
    continuation(ctx, scenes["cornell_box"], kernel, flags, seed=kernel * 16 + flags)


def test_continuation_on_large_scene_paths():
    """device-built threaded copies and the large-scene schedule, as test_views_on_large_scene_paths lowers them"""
    with capi.Context(0) as c:
        c.debug_limits(0, 0)
        sc = c.upload(util.scene("cornell_box_lens"))
        for kernel in KERNELS:
            for flags in (0, L.FLAG_WAVEFRONT):
                continuation(c, sc, kernel, flags, seed=100 + kernel)
        sc.release()


@pytest.mark.parametrize("flags", [0, L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_SERIAL,
                                   L.FLAG_STATS, L.FLAG_CULL])
@pytest.mark.parametrize("kernel", [L.KERNEL_GI, L.KERNEL_GI25, L.KERNEL_ACCUMULATOR, L.KERNEL_BASIC_CU])
def test_list_order_does_not_matter(ctx, scenes, kernel, flags):
    """the same mask rendered through its list in the compaction's order and reversed (lt_debug_ctx_list_order): the
    reversed list puts every warp's pixels in other lanes and other warps, the values stay bit for bit"""
    sc = scenes["cornell_box"]
    mask = random_mask(7 + kernel, 0.5)
    start = np.random.default_rng(3).random((H, W, 3), dtype=np.float32)
    p = capi.make_params(kernel, W, H, max_ray_depth=4, frames=5, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
    want = plain(ctx, sc, p, start, 6)
    a, a2 = masked(ctx, sc, p, nan_outside(start, mask), 6, mask, start)
    launches = ctx.stats().kernel_launches
    ctx.debug_list_order(True)
    try:
        b, b2 = masked(ctx, sc, p, nan_outside(start, mask), 6, mask, start)
        reversed_launches = ctx.stats().kernel_launches
        full, _ = masked(ctx, sc, p, start, 6)
    finally:
        ctx.debug_list_order(False)
    assert reversed_launches == launches + 1  # the reversal kernel
    what = "kernel %d, flags %d" % (kernel, flags)
    assert_masked(a, want, nan_outside(start, mask), mask, what + ", compaction order")
    util.assert_bit_equal(b, a, what + ", reversed list")
    util.assert_bit_equal(b2, a2, what + ", reversed list, m2")
    util.assert_bit_equal(full, want, what + ", NULL mask, reversed list")


def test_empty_mask_writes_nothing(ctx, scenes):
    empty = np.zeros((H, W), bool)
    start = nan_outside(np.zeros((H, W, 3), np.float32), empty)
    for flags in (0, L.FLAG_WAVEFRONT, L.FLAG_STATS):
        p = capi.make_params(L.KERNEL_GI, W, H, max_ray_depth=3, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
        got, got2 = masked(ctx, scenes["cornell_box"], p, start, 3, empty, start)
        util.assert_bit_equal(got, start, "out")
        util.assert_bit_equal(got2, start, "m2")
        s = ctx.stats()
        assert s.kernel_launches == 1 and s.rays == 0


def welford(samples):
    """the Welford order of lt_render_masked_device in float32, one rounding per operation"""
    mean = np.zeros_like(samples[0])
    m2 = np.zeros_like(samples[0])
    for n, x in enumerate(samples):
        if n == 0:
            mean, m2 = x.copy(), np.zeros_like(x)
            continue
        d = x - mean
        nf = np.float32(n)
        mean = (x + mean * nf) / np.float32(n + 1)
        m2 = m2 + d * (x - mean)
    return mean, m2


@pytest.mark.parametrize("flags", [L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT])
@pytest.mark.parametrize("kernel", [L.KERNEL_GI, L.KERNEL_ACCUMULATOR, L.KERNEL_GI25])
def test_m2_is_welford_of_the_frame_samples(ctx, scenes, kernel, flags):
    sc = scenes["cornell_box"]
    frames = 6
    one = capi.make_params(kernel, W, H, max_ray_depth=3, frames=1, accum_mode=L.ACCUM_NONE, flags=flags)
    zero = np.zeros((H, W, 3), np.float32)
    samples = [plain(ctx, sc, one, zero, n) for n in range(frames)]
    mean, m2 = welford(samples)
    p = capi.make_params(kernel, W, H, max_ray_depth=3, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
    got, got2 = masked(ctx, sc, p, zero, 0, None, zero)
    util.assert_bit_equal(got, mean, "running mean")
    util.assert_bit_equal(got2, m2, "m2")
    assert (m2 > 0).any()
    # in two calls: 2 frames, then 4 from frameCount 2
    p.frames = 2
    a, a2 = masked(ctx, sc, p, zero, 0, None, zero)
    p.frames = 4
    b, b2 = masked(ctx, sc, p, a, 2, np.ones((H, W), bool), a2)
    util.assert_bit_equal(b, mean, "running mean, two calls")
    util.assert_bit_equal(b2, m2, "m2, two calls")


def test_running_mean_against_the_oracle(ctx, scenes):
    """one small case: the masked running mean equals oracle.accumulate of the oracle's own frames"""
    sb = util.scene("cornell_box")
    w, h, frames = 48, 36, 4
    want = np.zeros((h, w, 3), np.float32)
    samples = []
    for n in range(frames):
        x = O.render(L.KERNEL_GI, sb, cam(n), w, h, max_ray_depth=3)
        samples.append(x)
        O.accumulate(want, x, n)
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=3, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN)
    zero = np.zeros((h, w, 3), np.float32)
    out = dev(zero)
    m2 = dev(zero)
    ctx.render_masked_device(scenes["cornell_box"], cam(0), p, out.data_ptr(), None, m2.data_ptr(), sync=True)
    util.assert_bit_equal(host(out), want, "running mean against the oracle")
    util.assert_bit_equal(host(m2), welford(samples)[1], "m2 of the oracle's frames")


@pytest.mark.parametrize("flags", [0, L.FLAG_WAVEFRONT])
def test_adaptive_loop(ctx, scenes, flags):
    """16 frames on every pixel, then three masked rounds of 16 on the pixels whose relative standard error stays above a
    threshold; every pixel ends bit for bit as a plain render of its own frame count"""
    sc = scenes["cornell_box"]
    zero = np.zeros((H, W, 3), np.float32)
    p = capi.make_params(L.KERNEL_GI, W, H, max_ray_depth=3, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
    out, m2 = dev(zero), dev(zero)
    n = torch.full((H, W), 16, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()  # torch's stream and the context's: the renders below are synchronous
    ctx.render_masked_device(sc, cam(0), p, out.data_ptr(), None, m2.data_ptr(), sync=True)
    sizes = []
    for rnd in range(3):
        nf = n.to(torch.float32)[..., None]
        err = torch.sqrt(m2 / (nf * (nf - 1))) / out.clamp_min(1e-3)
        mask = (err.amax(dim=2) > 0.05) & (n == 16 * (rnd + 1))
        sizes.append(int(mask.sum()))
        if sizes[-1] == 0:
            break
        m = mask.to(torch.uint8).contiguous()
        torch.cuda.synchronize()
        ctx.render_masked_device(sc, cam(16 * (rnd + 1)), p, out.data_ptr(), m.data_ptr(), m2.data_ptr(), sync=True)
        n += 16 * mask.to(torch.int32)
    torch.cuda.synchronize()
    assert sizes[0] > 0 and sizes == sorted(sizes, reverse=True), sizes
    counts = host(n)
    got = host(out)
    for k in np.unique(counts):
        q = capi.make_params(L.KERNEL_GI, W, H, max_ray_depth=3, frames=int(k), accum_mode=L.ACCUM_RUNNING_MEAN,
                             flags=flags)
        want = plain(ctx, sc, q, zero, 0)
        sel = counts == k
        util.assert_bit_equal(got[sel], want[sel], "pixels of %d frames" % k)


@pytest.mark.parametrize("flags", [L.FLAG_MEGAKERNEL, L.FLAG_WAVEFRONT, 0])
@pytest.mark.parametrize("kernel", [L.KERNEL_GI, L.KERNEL_BASIC_CU])
def test_stats_count_the_masked_pixels(ctx, scenes, kernel, flags):
    """the counters are per pixel: a mask's and its complement's add up to the full image's"""
    p = capi.make_params(kernel, W, H, max_ray_depth=3, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN,
                         flags=flags | L.FLAG_STATS)
    zero = np.zeros((H, W, 3), np.float32)
    mask = random_mask(11, 0.4)
    counts = []
    for m in (mask, ~mask, None):
        masked(ctx, scenes["cornell_box"], p, zero, 0, m)
        s = ctx.stats()
        counts.append(np.array([s.rays, s.node_tests, s.tri_tests], np.uint64))
    plain(ctx, scenes["cornell_box"], p, zero, 0)
    s = ctx.stats()
    assert (counts[2] == np.array([s.rays, s.node_tests, s.tri_tests], np.uint64)).all()
    assert (counts[0] + counts[1] == counts[2]).all() and counts[0][0] > 0


def test_errors_leave_the_outputs(ctx, scenes):
    sc = scenes["cornell_box"]
    lib = ctx.lib
    start = nan_outside(np.zeros((H, W, 3), np.float32), np.zeros((H, W), bool))
    out, m2 = dev(start), dev(start)
    mask = dev(np.ones((H, W), np.uint8))
    c = np.ascontiguousarray(cam(0), dtype=L.CAMERA)

    def call(p, mask_ptr=mask.data_ptr(), m2_ptr=m2.data_ptr()):
        return lib.lt_render_masked_device(ctx.h, sc.h, c.ctypes.data, C.byref(p), C.c_void_p(mask_ptr),
                                           C.c_void_p(out.data_ptr()), C.c_void_p(m2_ptr), 1)

    for mode in (L.ACCUM_NONE, L.ACCUM_WEIGHTED_SUM):
        assert call(capi.make_params(L.KERNEL_GI, W, H, accum_mode=mode)) == capi.ERR_INVALID
    assert call(capi.make_params(L.KERNEL_GI, W, H, accum_mode=L.ACCUM_RUNNING_MEAN, frame_stride=2)) == capi.ERR_INVALID
    assert b"device_m2" in lib.lt_last_error(ctx.h)
    host_mask = np.ones((H, W), np.uint8)
    good = capi.make_params(L.KERNEL_GI, W, H, max_ray_depth=3, accum_mode=L.ACCUM_RUNNING_MEAN)
    assert call(good, mask_ptr=host_mask.ctypes.data) == capi.ERR_INVALID
    assert b"device_mask is not device memory" in lib.lt_last_error(ctx.h)
    host_m2 = np.zeros((H, W, 3), np.float32)
    assert call(good, m2_ptr=host_m2.ctypes.data) == capi.ERR_INVALID
    assert call(good, m2_ptr=m2.data_ptr() + 2) == capi.ERR_INVALID  # not 4-byte aligned
    assert call(capi.make_params(L.KERNEL_GI, 0, H)) == capi.ERR_INVALID
    assert call(capi.make_params(99, W, H)) == capi.ERR_UNSUPPORTED
    assert call(capi.make_params(L.KERNEL_GI, W, H, frames=0)) == capi.ERR_INVALID
    torch.cuda.synchronize()
    util.assert_bit_equal(host(out), start, "out after the errors")
    util.assert_bit_equal(host(m2), start, "m2 after the errors")
    assert (host_m2 == 0).all()
    # the same arguments pass
    assert call(good) == 0


def test_images_above_int_max_pixels_are_refused(ctx, scenes):
    """a 50000 x 50000 image (2.5e9 pixels) is refused before anything is launched: the buffers stay as they were"""
    out = dev(np.full((4, 3), 7.0, np.float32))
    mask = dev(np.ones(16, np.uint8))
    c = np.ascontiguousarray(cam(0), dtype=L.CAMERA)
    for w, h in ((50000, 50000), (46341, 46341)):
        p = capi.make_params(L.KERNEL_GI, w, h, accum_mode=L.ACCUM_RUNNING_MEAN)
        for mask_ptr in (None, mask.data_ptr()):
            rc = ctx.lib.lt_render_masked_device(ctx.h, scenes["cornell_box"].h, c.ctypes.data, C.byref(p),
                                                 C.c_void_p(mask_ptr) if mask_ptr else None,
                                                 C.c_void_p(out.data_ptr()), C.c_void_p(out.data_ptr()), 1)
            assert rc == capi.ERR_UNSUPPORTED
            assert b"2^31 - 1 pixels" in ctx.lib.lt_last_error(ctx.h)
    torch.cuda.synchronize()
    assert (host(out) == 7.0).all()


def test_multi_gpu_context_is_unsupported():
    with util.device_group(max(2, min(torch.cuda.device_count(), 8))) as multi:
        sc = multi.upload(util.scene("cornell_box"))
        start = np.full((H, W, 3), 5.0, np.float32)
        out = dev(start)
        p = capi.make_params(L.KERNEL_GI, W, H, accum_mode=L.ACCUM_RUNNING_MEAN)
        with pytest.raises(capi.LtError, match="multi-GPU"):
            multi.render_masked_device(sc, cam(0), p, out.data_ptr())
        util.assert_bit_equal(host(out), start, "out after the refused call")
        sc.release()

"""The wavefront pipeline carries each path's state in its queue entry, beside the ray.  These cases reach what the
parity suite does not: queues filled to capacity, the bounce caps at both ends, and the 25-sample GI kernel over
several bounces.  In each, the wavefront image must equal the megakernel image bit for bit."""
import pytest

import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu

WAVEFRONT = [L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED]


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def cornell(ctx):
    sc = ctx.upload(util.scene("cornell_box"))
    yield sc
    sc.release()


def render(ctx, sc, cam, kernel, w, h, depth, frames, flags):
    ctx.accum_reset()
    return ctx.render(sc, cam, capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames,
                                                accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)).copy()


def assert_wavefront_equals_megakernel(ctx, sc, cam, kernel, w, h, depth, frames):
    want = render(ctx, sc, cam, kernel, w, h, depth, frames, L.FLAG_MEGAKERNEL)
    for flags in WAVEFRONT:
        got = render(ctx, sc, cam, kernel, w, h, depth, frames, flags)
        util.assert_bit_equal(got, want, "wavefront (flags %d) vs megakernel" % flags)


def test_camera_inside_the_box(ctx, cornell):
    """Every camera ray hits a wall, so every path of the batch emits a shadow ray and then an extension ray: both
    queues fill to capacity."""
    cam = L.make_camera(0, 2.5, 0.0, 0.0, 0)
    w, h = 192, 128
    _, hit, _ = ctx.primary_hits(cornell, cam, L.KERNEL_GI, w, h)
    assert hit.all()
    assert_wavefront_equals_megakernel(ctx, cornell, cam, L.KERNEL_GI, w, h, 4, 5)


@pytest.mark.parametrize("depth", [1, 32])
def test_bounce_caps(ctx, cornell, depth):
    assert_wavefront_equals_megakernel(ctx, cornell, util.default_camera(0.0, 2), L.KERNEL_GI, 128, 96, depth, 3)


def test_gi25_several_bounces(ctx, cornell):
    assert_wavefront_equals_megakernel(ctx, cornell, util.default_camera(0.03, 1), L.KERNEL_GI25, 64, 48, 4, 2)

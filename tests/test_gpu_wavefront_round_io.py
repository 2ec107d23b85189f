"""The wavefront pipeline compiles its shade kernel for each kind of round (first shadow rays, later shadow rays,
extension rays) and loads only what that kind reads: a shadow ray's hit travels as one word, and an extension entry
carries the cosine its light hit adds instead of its normal and direction.  Counting launches that retrace light hits
mix the kinds and keep the full entries.  In every case below the wavefront image equals the megakernel image bit for
bit, and the counting launches count what they counted before the round kinds existed."""
import pytest

import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu

WAVEFRONT = [L.FLAG_WAVEFRONT, L.FLAG_WAVEFRONT | L.FLAG_SERIAL, L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED]

INSIDE = L.make_camera(0, 2.5, 0.0, 0.0, 0)  # every camera ray hits a wall; the light is seen from every bounce

# (scene, camera, kernel, width, height, max_ray_depth, frames)
CASES = {
    "gi_depth1": ("cornell_box", util.default_camera(0.0, 1), L.KERNEL_GI, 96, 64, 1, 3),
    "gi_depth2": ("cornell_box", util.default_camera(0.0, 1), L.KERNEL_GI, 96, 64, 2, 3),
    "gi_depth4": ("cornell_box", util.default_camera(0.02, 3), L.KERNEL_GI, 96, 64, 4, 3),
    "gi_depth32": ("cornell_box", util.default_camera(0.0, 1), L.KERNEL_GI, 64, 48, 32, 2),
    "gi25": ("cornell_box", util.default_camera(0.03, 1), L.KERNEL_GI25, 48, 32, 3, 2),
    "accumulator": ("cornell_box", util.default_camera(0.0, 2), L.KERNEL_ACCUMULATOR, 96, 64, 0, 4),
    "basic_lighting": ("cornell_box", util.default_camera(0.0, 2), L.KERNEL_LIGHTING25, 48, 32, 0, 2),
    "lens_gi": ("cornell_box_lens", util.default_camera(0.01, 2), L.KERNEL_GI, 96, 64, 4, 3),
    "inside_gi": ("cornell_box", INSIDE, L.KERNEL_GI, 96, 64, 6, 3),
    "odd_size_gi": ("cornell_box", util.default_camera(0.0, 4), L.KERNEL_GI, 101, 67, 4, 3),
}

# Counters (rays, node tests, triangle tests) of wavefront launches with LT_FLAG_STATS (the reference's traversals:
# light hits retraced, so rounds mix kinds) and with LT_FLAG_STATS | LT_FLAG_STATS_TRACED (the rays the exact pipelines
# trace: homogeneous rounds), as the build before the round kinds counted them.
COUNTED = ("gi_depth4", "lens_gi", "inside_gi", "accumulator")
EXPECTED_COUNTS = {
    ('gi_depth4', False): (54559, 1509535, 146499),
    ('gi_depth4', True): (54437, 1504655, 146116),
    ('lens_gi', False): (47732, 1865516, 141365),
    ('lens_gi', True): (47663, 1862509, 141153),
    ('inside_gi', False): (146722, 5209740, 493930),
    ('inside_gi', True): (145201, 5147365, 489117),
    ('accumulator', False): (33012, 622728, 59378),
    ('accumulator', True): (33012, 622728, 59378),
}


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


def render(ctx, scenes, case, flags):
    name, cam, kernel, w, h, depth, frames = CASES[case]
    ctx.accum_reset()
    return ctx.render(scenes[name], cam, capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames,
                                                          accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)).copy()


def counts(ctx, scenes, case, flags):
    img = render(ctx, scenes, case, L.FLAG_WAVEFRONT | flags)
    st = ctx.stats()
    return img, (st.rays, st.node_tests, st.tri_tests)


@pytest.mark.parametrize("case", sorted(CASES))
def test_wavefront_equals_megakernel(ctx, scenes, case):
    want = render(ctx, scenes, case, L.FLAG_MEGAKERNEL)
    for flags in WAVEFRONT:
        util.assert_bit_equal(render(ctx, scenes, case, flags), want, "%s: wavefront (flags %d) vs megakernel"
                              % (case, flags))


def test_camera_inside_the_box_sees_only_surfaces(ctx, scenes):
    _, hit, _ = ctx.primary_hits(scenes["cornell_box"], INSIDE, L.KERNEL_GI, 96, 64)
    assert hit.all()


@pytest.mark.parametrize("case", COUNTED)
@pytest.mark.parametrize("traced", [False, True], ids=["stats", "stats_traced"])
def test_counting_launches(ctx, scenes, case, traced):
    flags = L.FLAG_STATS | (L.FLAG_STATS_TRACED if traced else 0)
    img, got = counts(ctx, scenes, case, flags)
    util.assert_bit_equal(img, render(ctx, scenes, case, L.FLAG_MEGAKERNEL), "%s: counting launch vs megakernel" % case)
    assert got == EXPECTED_COUNTS[(case, traced)]

"""The launch plan (lt_debug_plan, no device needed): which pipeline, tree, batching and sizes lt_render chooses for a
launch.  Device: 180 GiB and 148 SMs (a B200).  Scenes: the 83-node Cornell box (host-built threaded copies) and the
1 999 419-node tree of the 1 M-triangle mesh (device-built copies); their stack depths are fixed here at 8 and 40
levels, which only the shared-memory sizes depend on."""
import pytest

from lens_trace_b200 import capi, layouts as L
from lens_trace_b200.capi import (PIPE_FLAT, PIPE_FLAT_STREAM, PIPE_PATH, PIPE_WAVEFRONT, TREE_CHILD_PAIR,
                                  TREE_DEVICE_THREADED, TREE_HOST_THREADED)

B200 = dict(total_mem=180 << 30, sm_count=148)
SMALL = dict(node_count=83, stack_depth=8)
LARGE = dict(node_count=1999419, stack_depth=40)
HUGE = dict(node_count=20000000, stack_depth=40)  # 8 threaded copies would take 5.1 GB: none are made

# dynamic shared memory: (stack levels x (2 when culled) + 16 list entries) x 128 threads x 4 bytes
SMEM_SMALL, SMEM_SMALL_CULL, SMEM_LARGE, SMEM_LARGE_CULL = 12288, 16384, 28672, 49152
SMEM_THREADED = 8192


def plan(kernel, w, h, frames=1, flags=0, scene=SMALL, max_ray_depth=0):
    p = capi.make_params(kernel, w, h, frames=frames, flags=flags, max_ray_depth=max_ray_depth)
    return capi.plan(p, scene["node_count"], scene["stack_depth"], B200["total_mem"], B200["sm_count"])


def check(got, **want):
    assert got["error"] == 0, got["message"]
    assert {k: got[k] for k in want} == want


def test_gi_default_schedule_small_scene():
    got = plan(L.KERNEL_GI, 1920, 1080, frames=64)
    check(got, pipeline=PIPE_WAVEFRONT, tree=TREE_HOST_THREADED, stats=0, cull=0, batch_frames=16, streams=2,
          rounds=34, samples_per_frame=1, shared_primary=1, classify=1, smem_stack=SMEM_SMALL,
          smem_trace=SMEM_THREADED, blocks_per_sm=8, grid=148 * 8)
    # two workspaces of 16 x 2 073 600 paths at 184 B (+ padding), and the per-pixel primary records
    assert got["workspace_bytes"] == 2 * 6104682752 + 60136704


def test_gi_wavefront_starts_at_two_to_the_23_paths():
    check(plan(L.KERNEL_GI, 1920, 1080, frames=4), pipeline=PIPE_PATH, tree=TREE_HOST_THREADED)  # 8 294 400 paths
    check(plan(L.KERNEL_GI, 1920, 1080, frames=5), pipeline=PIPE_WAVEFRONT, tree=TREE_HOST_THREADED, batch_frames=3,
          streams=2)


def test_gi_stats_and_serial():
    check(plan(L.KERNEL_GI, 1920, 1080, frames=64, flags=L.FLAG_STATS), pipeline=PIPE_WAVEFRONT, tree=TREE_CHILD_PAIR,
          stats=1, batch_frames=16, streams=1, shared_primary=0, classify=0, smem_trace=SMEM_SMALL, blocks_per_sm=8)
    # one stream: 32 frames fit 2^26 paths, capped at 16 by the 25-bit path id
    check(plan(L.KERNEL_GI, 1920, 1080, frames=64, flags=L.FLAG_SERIAL), pipeline=PIPE_WAVEFRONT,
          tree=TREE_HOST_THREADED, batch_frames=16, streams=1, shared_primary=1, classify=1)


def test_gi_4k_five_frames_large_scene():
    check(plan(L.KERNEL_GI, 3840, 2160, frames=5, scene=LARGE), pipeline=PIPE_WAVEFRONT, tree=TREE_CHILD_PAIR,
          batch_frames=3, streams=2, smem_stack=SMEM_LARGE, smem_trace=SMEM_LARGE, blocks_per_sm=7, grid=148 * 7)


def test_accumulator():
    check(plan(L.KERNEL_ACCUMULATOR, 1920, 1080, frames=16), pipeline=PIPE_PATH, tree=TREE_HOST_THREADED)
    check(plan(L.KERNEL_ACCUMULATOR, 1920, 1080, frames=17), pipeline=PIPE_WAVEFRONT, tree=TREE_HOST_THREADED,
          rounds=2, samples_per_frame=1, classify=1)
    # coherent rays on the megakernel: a large scene's device-built copies
    check(plan(L.KERNEL_ACCUMULATOR, 1920, 1080, scene=LARGE), pipeline=PIPE_PATH, tree=TREE_DEVICE_THREADED)
    check(plan(L.KERNEL_ACCUMULATOR, 1920, 1080, scene=HUGE), pipeline=PIPE_PATH, tree=TREE_CHILD_PAIR)
    check(plan(L.KERNEL_ACCUMULATOR, 1920, 1080, flags=L.FLAG_WAVEFRONT, scene=LARGE), pipeline=PIPE_WAVEFRONT,
          tree=TREE_CHILD_PAIR)


@pytest.mark.parametrize("scene", [SMALL, LARGE])
@pytest.mark.parametrize("kernel", [L.KERNEL_LIGHTING25, L.KERNEL_GI25])
def test_25_sample_kernels_stay_on_the_megakernel(kernel, scene):
    check(plan(kernel, 1920, 1080, frames=64, scene=scene), pipeline=PIPE_PATH)
    check(plan(kernel, 1920, 1080, frames=64, flags=L.FLAG_WAVEFRONT, scene=scene), pipeline=PIPE_WAVEFRONT,
          samples_per_frame=25, classify=0, shared_primary=1)


def test_forced_wavefront_limits():
    check(plan(L.KERNEL_GI, 1920, 1080, frames=64, max_ray_depth=32, flags=L.FLAG_WAVEFRONT), pipeline=PIPE_WAVEFRONT,
          rounds=66)
    check(plan(L.KERNEL_GI, 1920, 1080, frames=64, max_ray_depth=33), pipeline=PIPE_PATH)
    got = plan(L.KERNEL_GI, 1920, 1080, frames=64, max_ray_depth=33, flags=L.FLAG_WAVEFRONT)
    assert got["error"] == capi.ERR_UNSUPPORTED
    assert got["message"] == "lt_render: the wavefront pipeline handles max_ray_depth <= 32 (use the default schedule)"
    check(plan(L.KERNEL_GI, 8192, 4096, flags=L.FLAG_WAVEFRONT), pipeline=PIPE_WAVEFRONT, batch_frames=1, streams=1)
    check(plan(L.KERNEL_GI, 8192, 4097), pipeline=PIPE_PATH)
    got = plan(L.KERNEL_GI, 8192, 4097, flags=L.FLAG_WAVEFRONT)
    assert got["error"] == capi.ERR_UNSUPPORTED
    assert got["message"] == "lt_render: the wavefront pipeline handles at most 2^25 pixels per frame"


@pytest.mark.parametrize("scene,smem", [(SMALL, SMEM_SMALL_CULL), (LARGE, SMEM_LARGE_CULL)])
def test_cull(scene, smem):
    check(plan(L.KERNEL_GI, 1920, 1080, flags=L.FLAG_CULL, scene=scene), pipeline=PIPE_WAVEFRONT,
          tree=TREE_CHILD_PAIR, cull=1, smem_stack=smem, shared_primary=0, classify=0)
    check(plan(L.KERNEL_GI, 1920, 1080, flags=L.FLAG_CULL | L.FLAG_MEGAKERNEL, scene=scene), pipeline=PIPE_PATH,
          tree=TREE_CHILD_PAIR, cull=1, smem_stack=smem)


def test_deterministic_kernels():
    # 240 x 270 tiles of 8 x 4 pixels, 4 warps a block: 16 200 blocks of work; 120 x 135 blocks of 16 x 8 pixels
    check(plan(L.KERNEL_BASIC_CU, 1920, 1080, scene=LARGE), pipeline=PIPE_FLAT_STREAM, tree=TREE_CHILD_PAIR,
          blocks_per_sm=7, grid=148 * 7)
    for flags in (L.FLAG_NO_STREAM, L.FLAG_STATS, L.FLAG_CULL):
        check(plan(L.KERNEL_BASIC_CU, 1920, 1080, flags=flags, scene=LARGE), pipeline=PIPE_FLAT,
              tree=TREE_CHILD_PAIR, grid=16200)
    check(plan(L.KERNEL_BASIC_CU, 1920, 1080), pipeline=PIPE_FLAT, tree=TREE_HOST_THREADED)
    check(plan(L.KERNEL_BASIC_CU, 1920, 1080, flags=L.FLAG_NO_THREADED), pipeline=PIPE_FLAT, tree=TREE_CHILD_PAIR)
    check(plan(L.KERNEL_CUSTOM_BARY, 7, 3, scene=LARGE), pipeline=PIPE_FLAT_STREAM, grid=1)


def test_invalid_params_are_rejected():
    with pytest.raises(capi.LtError):
        plan(L.KERNEL_GI, 0, 1080)

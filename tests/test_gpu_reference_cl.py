"""GPU vs the reference's OWN OpenCL kernel text (oracle/_ref/libltref_cl.so: the .cl files compiled for the
CPU through oracle/cl_shim, built where /root/reference exists and shipped to the GPU box).

The CUDA path is bit-identical to the restatement in LTO_FP_DEVICE mode (tests/test_gpu_parity.py) and the
restatement in LTO_FP_PLAIN mode is bit-identical to this library (tests/test_oracle_cl.py).  This file closes
the triangle directly: CUDA image vs reference-text image.  The two differ only by what OpenCL C leaves to the
implementation (fusing inside dot/cross, cosf/sinf), i.e. by last-place rounding -- which moves a handful of
edge pixels to another triangle and, downstream of a flipped 8-bit hash value, to another light sample.  Bounds
(north star: 1e-4 relative per pixel for deterministic passes, RMSE/PSNR for converged stochastic GI):
  * deterministic kernels: >= 99.8 % of pixels within 1e-4 relative
  * one stochastic sample: >= 99.5 % of pixels within 1e-4 relative
  * 64-frame running mean: PSNR >= 36 dB against the reference-text mean (measured ~40 dB; the residue is the
    ~0.1 % edge pixels whose primary hit differs in every frame).

Without that library the live tests skip; the reference-text images stored in tests/golden/ref_cl_*.npz keep the
CUDA path compared with the reference's kernel text under the same bounds."""
import glob
import os

import numpy as np
import pytest

import lt_oracle as O
import lt_ref_cl as R
import util
from lens_trace_b200 import capi, layouts as L

pytestmark = pytest.mark.gpu
needs_ref_cl = pytest.mark.skipif(not R.available(), reason="oracle/_ref/libltref_cl.so not shipped")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def frac_within(got, want):
    return float(np.isclose(got, want, rtol=1e-4, atol=1e-6).all(axis=-1).mean())


@needs_ref_cl
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens", "green_wall"])
@pytest.mark.parametrize("kernel", [L.KERNEL_BASIC_CL, L.KERNEL_CUSTOM_BARY])
def test_deterministic_kernels_vs_reference_text(ctx, name, kernel):
    sb = util.scene(name)
    sc = ctx.upload(sb)
    cam = util.default_camera(0.01)
    got = ctx.render(sc, cam, capi.make_params(kernel, 200, 150))
    want = R.render(kernel, sb, cam, 200, 150)
    sc.release()
    assert frac_within(got, want) >= 0.998


@needs_ref_cl
@pytest.mark.parametrize("name", ["cornell_box", "cornell_box_lens"])
@pytest.mark.parametrize("kernel,depth", [(L.KERNEL_ACCUMULATOR, 16), (L.KERNEL_GI, 4), (L.KERNEL_GI, 16)])
@pytest.mark.parametrize("mode", [0, 1])
def test_one_stochastic_sample_vs_reference_text(ctx, kernel, depth, mode, name):
    sb = util.scene(name)
    sc = ctx.upload(sb)
    for frame in (0, 3, 40):
        cam = util.default_camera(0.0, frame)
        got = ctx.render(sc, cam, capi.make_params(kernel, 160, 120, kernel_mode=mode, max_ray_depth=depth))
        want = R.render(kernel, sb, cam, 160, 120, kernel_mode=mode, max_ray_depth=depth)
        assert frac_within(got, want) >= 0.995, (kernel, frame)
    sc.release()


@needs_ref_cl
@pytest.mark.parametrize("kernel,depth", [(L.KERNEL_GI, 4), (L.KERNEL_ACCUMULATOR, 16)])
def test_converged_running_mean_vs_reference_text(ctx, kernel, depth):
    # the example protocol (examples/global_illumination/src/main.cpp:296-325): frameCount 0..63, running mean
    sb = util.scene("cornell_box")
    sc = ctx.upload(sb)
    w, h, frames = 160, 120, 64
    ctx.accum_reset()
    got = ctx.render(sc, util.default_camera(0.0, 0),
                     capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN))
    sc.release()
    acc = np.zeros((h, w, 3), np.float32)
    for f in range(frames):
        O.accumulate(acc, R.render(kernel, sb, util.default_camera(0.0, f), w, h, max_ray_depth=depth), f)
    mse = float(((got.astype(np.float64) - acc) ** 2).mean())
    psnr = 10.0 * np.log10(1.0 / mse)
    assert psnr >= 36.0, psnr
    assert frac_within(got, acc) >= 0.95  # a pixel leaves 1e-4 if any one of its 64 samples took another branch


# the bounds above: deterministic kernels, then one stochastic sample (the 25-sample files are not covered here)
GOLDEN_BOUND = {L.KERNEL_BASIC_CL: 0.998, L.KERNEL_CUSTOM_BARY: 0.998, L.KERNEL_ACCUMULATOR: 0.995, L.KERNEL_GI: 0.995}


@pytest.mark.parametrize("path", sorted(p for p in glob.glob(os.path.join(util.GOLDEN, "ref_cl_*.npz"))
                                        if int(np.load(p)["kernel"]) in GOLDEN_BOUND),
                         ids=lambda p: os.path.basename(p)[7:-4])
def test_cuda_path_vs_reference_cl_golden(ctx, path):
    """Images the reference's kernel text computed (stored with the buffers and cameras they were made with):
    the CUDA path renders every case within the bound of its kind."""
    g = np.load(path)
    sb = L.SceneBuffers(g["nodes"], g["prims"], g["materials"], g["lights"])
    kernel, w, h = int(g["kernel"]), int(g["width"]), int(g["height"])
    sc = ctx.upload(sb)
    for i in range(len(g["color"])):
        cam = util.default_camera(float(g["yaw"][i]), int(g["frame_count"][i]))
        got = ctx.render(sc, cam, capi.make_params(kernel, w, h, kernel_mode=int(g["mode"][i]),
                                                    max_ray_depth=int(g["max_ray_depth"][i])))
        assert frac_within(got, g["color"][i]) >= GOLDEN_BOUND[kernel], (os.path.basename(path), i)
    sc.release()
